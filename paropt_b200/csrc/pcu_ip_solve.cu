// pcu_ip_solve.cu -- KKT set-up / solve, step statistics, starting point and the
// major loop of the CUDA-resident interior-point core (second half of pcu_ip).
#include <math.h>
#include <string.h>

#include <algorithm>

#include "pcu_ip.cuh"
#include "pcu_wide.cuh"

int pcu_mdot_enqueue(pcu_ctx *ctx, const double *x, const ColTable &cols,
                     int ncols, long long n, int dst_off);
int pcu_gram_enqueue(pcu_ctx *ctx, const ColTable &cols, int m,
                     const double *Dinv, const double *Cw, const WDesc &wd,
                     long long n, int *ld_out, const double *d2 = nullptr,
                     int rhs_col = -1);

#define launch_tile pcu_launch_tile
static const RedBuf NO_RED = {nullptr, nullptr, nullptr, 0};

// LS flags (IP.h:220-225)
enum {
  LS_SUCCESS = 1,
  LS_FAILURE = 2,
  LS_MIN_STEP = 4,
  LS_MAX_ITERS = 8,
  LS_NO_IMPROVEMENT = 16,
  LS_SHORT_STEP = 32
};
enum { BS_MONOTONE = 0, BS_MEHROTRA = 1, BS_MPC = 2, BS_COMP_FRACTION = 3 };

// ------------------------------------------------------- setUpKKTDiagSystem
// IP.cpp:1832-1930 (diagonal + Ew factor; G follows in setUpKKTSystem)
int pcu_ip::setUpKKTDiagSystem(Vars &vars, int use_qn, int identity) {
  pass1_ready = 0;
  auto launch = [&](auto f) -> int {
    f.v = vars.dv();
    f.lb = lb->d;
    f.ub = ub->d;
    f.Dinv = Dinv->d;
    f.Cw = Cw->d;
    double b0 = 0.0;
    if (qn && use_qn) b0 = qn->b0;
    b0_used = b0;
    f.b0sig = b0 + opt.qn_sigma;
    f.identity = identity;
    f.small_ = 1e-4;
    f.k = kconst();
    return launch_tile(ctx, f, nvars, wd, NO_RED);
  };
  // use_diag_hessian: diag(h) is the Hessian where the loop takes one (use_qn), as the
  // quasi-Newton b0 is: D0 = h + sigma + bound terms
  if (opt.use_diag_hessian && use_qn && !identity) {
    DiagHF f;
    f.h = hdiag->d;
    return launch(f);
  }
  return launch(DiagF());
}

// setUpKKTDiagSystem + the right-hand side (d1, d2) of the iteration's first
// diagonal solve, whose block part and reductions then ride in the Gram pass
// (setUpKKTSystem with_rhs).
int pcu_ip::setUpKKTDiagRhs(Vars &vars, int use_qn, double mu) {
  pass1_ready = 0;
  auto launch = [&](auto f) -> int {
    f.v = vars.dv();
    f.lb = lb->d;
    f.ub = ub->d;
    f.g = g->d;
    f.Dinv = Dinv->d;
    f.Cw = Cw->d;
    f.d1 = d1->d;
    f.d2 = d2->d;
    f.ncon = ncon;
    for (int j = 0; j < ncon; j++) {
      f.Acol.p[j] = Ac[j]->d;
      f.z.v[j] = vars.z[j];
    }
    if (gaz_valid && &vars == &variables) {
      // g - A z of this very point was left by the last update pass
      f.g = gaz->d;
      f.ncon = 0;
    }
    double b0 = 0.0;
    if (qn && use_qn) b0 = qn->b0;
    b0_used = b0;
    f.b0sig = b0 + opt.qn_sigma;
    f.mu = mu;
    f.k = kconst();
    return launch_tile(ctx, f, nvars, wd, NO_RED);
  };
  if (opt.use_diag_hessian && use_qn) {  // D0 = h + sigma + bound terms
    DiagRhsHF f;
    f.h = hdiag->d;
    return launch(f);
  }
  return launch(DiagRhsF());
}

// ----------------------------------------------------------- setUpKKTSystem
// One weighted Gram pass S = [A|Z]^T D0^-1 [A|Z] gives
//   G  = C0 + S_AA                                  (IP.cpp:1932-1969)
//   Ce = S_ZZ - S_ZA G^-1 S_AZ - M / (d d^T)        (IP.cpp:2646-2664)
// (pcu_dense_setup, into dense_host).  gdiag: diagonal added to G (s/zs + t/zt, or
// `small` for the least-squares start); NULL means s/zs + t/zt of `vars`.
int pcu_ip::setUpKKTSystem(Vars &vars, int use_qn, const double *gdiag,
                           int with_rhs) {
  const int q = (qn && use_qn) ? qn->size() : 0;
  const int m = ncon + q;
  ColTable V;
  for (int j = 0; j < ncon; j++) V.p[j] = Ac[j]->d;
  if (q > 0) qn->z_table(V, ncon);
  int ld = 0;
  if (m > 0) {
    if (with_rhs) {
      // column m = d1 of the first solve: row m of S is [A|Z]^T t1
      V.p[m] = d1->d;
      if (pcu_gram_enqueue(ctx, V, m + 1, Dinv->d, Cw->d, wd, nvars, &ld, d2->d, m))
        return 1;
    } else {
      if (pcu_gram_enqueue(ctx, V, m, Dinv->d, Cw->d, wd, nvars, &ld)) return 1;
    }
  }
  const DenseOff o = pcu_dense_offsets(ncon, q, ld);
  if (denseReserve(o)) return 1;
  dense_off = o;
  double *h = dense_host;
  if (m > 0) {
    if (ctx->big_fetch((size_t)ld * ld, h + o.S)) return 1;
    if (with_rhs) {
      pass1_r.resize(m);
      for (int j = 0; j < m; j++) pass1_r[j] = h[o.S + m + (size_t)ld * j];
      pass1_ready = 1;
    }
  }
  densePack(o, vars, barrier_param, gdiag);
  std::vector<double> scratch(PCU_DENSE_SCRATCH(ncon, q));
  pcu_dense_setup(h, o, scratch.data());
  return 0;
}

// dense_host large enough for the layout `o` (its contents are lost when it grows).  It is
// sized once for the widest solve the quasi-Newton object allows.  dense_dev follows it:
// kktChain allocates it again when the device runs the dense algebra.
int pcu_ip::denseReserve(const DenseOff &o) {
  if (dense_host && dense_cap >= o.total) return 0;
  if (dense_dev) cudaFree(dense_dev);
  if (dense_host) cudaFreeHost(dense_host);
  dense_dev = nullptr;
  dense_host = nullptr;
  const int qmax = qn ? qn->max_size() : 0;
  dense_cap = pcu_dense_offsets(ncon, qmax, 8 * ((ncon + qmax + 1 + 7) / 8)).total + 64;
  if (dense_cap < o.total) dense_cap = o.total + 64;
  PCU_CUDA_OK(cudaMallocHost(&dense_host, sizeof(double) * dense_cap));
  return 0;
}

// The inputs of the dense algebra at `vars` into dense_host, laid out by `o`.  gdiag (the
// least-squares start's G = gdiag I + A^T D0^-1 A) is packed as s = gdiag, zs = 1, t = 0,
// zt = 1: pcu_dense_setup's s/zs + t/zt is then gdiag exactly, and nothing else of that
// setup reads the dense inputs.
void pcu_ip::densePack(const DenseOff &o, const Vars &vars, double mu, const double *gdiag) {
  double *h = dense_host;
  h[o.mu] = mu;
  h[o.mu + 1] = 0.0;
  for (int i = 0; i < ncon; i++) {
    h[o.vz + i] = vars.z[i];
    h[o.vs + i] = gdiag ? gdiag[i] : vars.s[i];
    h[o.vt + i] = gdiag ? 0.0 : vars.t[i];
    h[o.vzs + i] = gdiag ? 1.0 : vars.zs[i];
    h[o.vzt + i] = gdiag ? 1.0 : vars.zt[i];
    h[o.cc + i] = c[i];
    h[o.gs + i] = gamma_s[i];
    h[o.gt + i] = gamma_t[i];
  }
  const int q = o.q;
  if (q > 0) {
    memcpy(h + o.M, qn->M.data(), sizeof(double) * q * q);
    memcpy(h + o.d0, qn->d0.data(), sizeof(double) * q);
    memcpy(h + o.Mf, qn->Mf.data(), sizeof(double) * q * q);
    memcpy(h + o.mpiv, qn->piv.data(), sizeof(double) * q);
  }
}

// ------------------------------------------------------------ computeKKTStep
// IP.cpp:2700-2737 with both inner diagonal solves (IP.cpp:2074-2243 and
// 2257-2369) merged: pass 1 -> reductions -> dense solves -> pass 2.
// VTp (optional, ncon + qn->size() values): [A | Z]^T of the (accumulated) step.
int pcu_ip::computeKKTStep(Vars &vars, Vars &b, Vars &y, int use_qn,
                           int accumulate, double *VTp, int emit_res,
                           double mu_res, int *emitted, int rhs_from_vars,
                           double stats_tau) {
  if (emitted) *emitted = 0;
  stats_ready = 0;
  {
    // The residual-free first solve needs the fused pass-1 / pass-2 kernels;
    // otherwise materialise the right-hand side first.
    const int q0 = denseWidth(use_qn);
    // more than 32 columns: only with this solve's first half already done by the
    // Gram pass (pass 2 is then Pass2RF, which takes any width)
    const bool fused_ok = emit_res && VTp && !force_direct_dots &&
                          q0 == (qn ? qn->size() : 0) && ncon + q0 > 0 &&
                          (ncon + q0 <= 32 || pass1_ready);
    if (rhs_from_vars && !fused_ok) {
      if (computeKKTRes(vars, mu_res, b, nullptr, nullptr, nullptr, 1)) return 1;
      rhs_from_vars = 0;
    }
    if (rhs_from_vars) denseResidual(vars, mu_res, b, nullptr, nullptr);
  }
  if (!dense_host) return 1;  // no setup yet
  const int q = denseWidth(use_qn);
  const int m = ncon + q;
  const IPConst k = kconst();
  ColTable V;
  for (int j = 0; j < ncon; j++) V.p[j] = Ac[j]->d;
  if (q > 0) qn->z_table(V, ncon);
  std::vector<double> r(m > 0 ? m : 1, 0.0);
  auto fused_pass1 = [&](auto f1) -> int {
    f1.v = vars.dv();
    f1.b = b.dv();
    f1.lb = lb->d;
    f1.ub = ub->d;
    f1.Dinv = Dinv->d;
    f1.Cw = Cw->d;
    f1.d1 = d1->d;
    f1.d2 = d2->d;
    f1.V = V;
    f1.m = m;
    f1.k = k;
    RedBuf rb = ctx->redbuf(decltype(f1)::NS, 0, 0);
    if (launch_tile(ctx, f1, nvars, wd, rb)) return 1;
    double out[decltype(f1)::NS];
    if (ctx->fetch(out)) return 1;
    for (int i = 0; i < m; i++) r[i] = out[i];
    return 0;
  };
  auto vars_pass1 = [&](auto f1) -> int {
    f1.v = vars.dv();
    f1.lb = lb->d;
    f1.ub = ub->d;
    f1.g = g->d;
    f1.Dinv = Dinv->d;
    f1.Cw = Cw->d;
    f1.d1 = d1->d;
    f1.d2 = d2->d;
    f1.V = V;
    f1.m = m;
    f1.ncon = ncon;
    for (int j = 0; j < ncon; j++) f1.z.v[j] = vars.z[j];
    f1.mu = mu_res;
    f1.k = k;
    RedBuf rb = ctx->redbuf(decltype(f1)::NS, 0, 0);
    if (launch_tile(ctx, f1, nvars, wd, rb)) return 1;
    double out[decltype(f1)::NS];
    if (ctx->fetch(out)) return 1;
    for (int i = 0; i < m; i++) r[i] = out[i];
    return 0;
  };
  if (pass1_ready) {
    // the previous (fused) pass 2 already did this solve's first half
    pass1_ready = 0;
    if ((int)pass1_r.size() != m) return 1;
    r = pass1_r;
    if (m == 0) r.assign(1, 0.0);
  } else if (rhs_from_vars) {
    if (m <= 8) {
      if (vars_pass1(Pass1VF<8>())) return 1;
    } else if (m <= 16) {
      if (vars_pass1(Pass1VF<16>())) return 1;
    } else if (m <= 24) {
      if (vars_pass1(Pass1VF<24>())) return 1;
    } else {
      if (vars_pass1(Pass1VF<32>())) return 1;
    }
  } else if (m > 0 && m <= 8) {
    if (fused_pass1(Pass1RF<8>())) return 1;
  } else if (m <= 16 && m > 0) {
    if (fused_pass1(Pass1RF<16>())) return 1;
  } else if (m <= 24 && m > 0) {
    if (fused_pass1(Pass1RF<24>())) return 1;
  } else if (m <= 32 && m > 0) {
    if (fused_pass1(Pass1RF<32>())) return 1;
  } else {
    Pass1F f1;
    f1.v = vars.dv();
    f1.b = b.dv();
    f1.lb = lb->d;
    f1.ub = ub->d;
    f1.Dinv = Dinv->d;
    f1.Cw = Cw->d;
    f1.d1 = d1->d;
    f1.d2 = d2->d;
    f1.t1 = t1->d;
    f1.k = k;
    if (launch_tile(ctx, f1, nvars, wd, NO_RED)) return 1;
    if (m > 0) {
      if (pcu_mdot_enqueue(ctx, t1->d, V, m, nvars, 0)) return 1;
      if (ctx->big_fetch(m, r.data())) return 1;
    }
  }
  // dense solves (IP.cpp:2150-2170, 2716-2722, 2288-2306): pcu_dense_step with the
  // factors of the last setup, at this solve's width
  DenseOff o = dense_off;
  o.q = q;
  o.m = m;
  double *h = dense_host;
  densePack(o, vars, mu_res, nullptr);
  for (int i = 0; i < ncon; i++) {
    h[o.bz + i] = b.z[i];
    h[o.bs + i] = b.s[i];
    h[o.bt + i] = b.t[i];
    h[o.bzs + i] = b.zs[i];
    h[o.bzt + i] = b.zt[i];
    if (accumulate) {
      h[o.yz + i] = y.z[i];
      h[o.ys + i] = y.s[i];
      h[o.yt + i] = y.t[i];
      h[o.yzs + i] = y.zs[i];
      h[o.yzt + i] = y.zt[i];
    }
  }
  for (int i = 0; i < m; i++) {
    h[o.r + i] = r[i];
    h[o.vtp + i] = accumulate && VTp ? VTp[i] : 0.0;
  }
  std::vector<double> scratch(PCU_DENSE_SCRATCH(ncon, q));
  pcu_dense_step(h, o, accumulate, h + o.coef, scratch.data());
  Pass2F f2;
  for (int j = 0; j < m; j++) f2.alpha.v[j] = h[o.coef + j];
  for (int i = 0; i < ncon; i++) {
    y.z[i] = h[o.yz + i];
    y.s[i] = h[o.ys + i];
    y.t[i] = h[o.yt + i];
    y.zs[i] = h[o.yzs + i];
    y.zt[i] = h[o.yzt + i];
  }
  f2.v = vars.dv();
  f2.b = b.dv();
  f2.y = y.dv();
  f2.lb = lb->d;
  f2.ub = ub->d;
  f2.Dinv = Dinv->d;
  f2.Cw = Cw->d;
  f2.d1 = d1->d;
  f2.d2 = d2->d;
  f2.V = V;
  f2.ncols = m;
  f2.accumulate = accumulate;
  f2.k = k;
  // [A | Z]^T p.  When the Gram pass covered every quasi-Newton vector the
  // products follow from linearity, [A|Z]^T D0^-1 (d1 + V alpha) = r + S alpha
  // (pcu_dense_step), without touching the N-vectors again.
  const int qa = qn ? qn->size() : 0;
  const bool derived = (q == qa) && !force_direct_dots;
  if (VTp && derived)
    for (int i = 0; i < m; i++) VTp[i] = h[o.vtp + i];
  if (emit_res && VTp && derived) {
    // pass 2 also writes the refinement residual (computeKKTRes +
    // addKKTResStep at the accumulated step) into `b`
    Pass2RF fr;
    fr.v = f2.v;
    fr.b = f2.b;
    fr.y = f2.y;
    fr.lb = f2.lb;
    fr.ub = f2.ub;
    fr.Dinv = f2.Dinv;
    fr.Cw = f2.Cw;
    fr.d1 = f2.d1;
    fr.d2 = f2.d2;
    fr.g = g->d;
    fr.V = V;
    fr.alpha = f2.alpha;
    fr.ncols = m;
    fr.accumulate = accumulate;
    fr.from_vars = rhs_from_vars;
    fr.mu_rhs = mu_res;
    fr.k = k;
    fr.mu = mu_res;
    fr.b0sig = opt.qn_sigma;
    for (int j = 0; j < ncon; j++) fr.beta.v[j] = vars.z[j] + y.z[j];
    for (int j = 0; j < q; j++) fr.beta.v[ncon + j] = 0.0;
    if (qn && !opt.sequential_linear_method) {  // IP.cpp:1474-1476
      fr.b0sig += qn->b0;
      if (q > 0) {
        std::vector<double> kap(q);
        qn->solve_compact(VTp + ncon, kap.data());
        for (int j = 0; j < q; j++) fr.beta.v[ncon + j] = kap[j];
      }
    }
    if (m <= 32 && !opt_no_fuse21) {
      // ... and the first half of the refinement solve on that residual
      auto fused21 = [&](auto ff) -> int {
        ff.v = fr.v; ff.b = fr.b; ff.y = fr.y;
        ff.lb = fr.lb; ff.ub = fr.ub; ff.Dinv = fr.Dinv; ff.Cw = fr.Cw;
        ff.d1 = fr.d1; ff.g = fr.g;
        ff.d2 = d2->d;
        ff.d1out = t1->d;
        ff.V = fr.V; ff.alpha = fr.alpha; ff.beta = fr.beta;
        ff.ncols = m; ff.accumulate = accumulate; ff.from_vars = fr.from_vars;
        ff.b0sig = fr.b0sig; ff.mu = fr.mu; ff.mu_rhs = fr.mu_rhs; ff.k = k;
        ff.cbank = -1;
        ff.apz = apz_target(accumulate, true);
        ff.nca = ncon;
        RedBuf rb = ctx->redbuf(decltype(ff)::NS, 0, 0);
        if (launch_tile(ctx, ff, nvars, wd, rb)) return 1;
        apz_done(accumulate, ff.apz);
        double out[decltype(ff)::NS];
        if (ctx->fetch(out)) return 1;
        pass1_r.assign(out, out + m);
        return 0;
      };
      int rc;
      if (m <= 8) rc = fused21(Pass2R1F<8>());
      else if (m <= 16) rc = fused21(Pass2R1F<16>());
      else if (m <= 24) rc = fused21(Pass2R1F<24>());
      else rc = fused21(Pass2R1F<32>());
      if (rc) return 1;
      std::swap(d1, t1);  // the next pass 2 reads d1' where the fused pass wrote it
      pass1_ready = 1;
    } else {
      // more than 32 columns: the same fusion on the column-split staged kernel
      // (whole 64-row tiles, no weighting constraints); otherwise the register-fed
      // Pass2RF and, in the next solve, Pass1F + a multi-dot
      int rc = -1;
      double *apz_w = apz_target(accumulate, true);
      if (!opt_no_fuse21 && !opt_no_wide) {
        Pass2R1F<0, 1> ff;
        ff.v = fr.v; ff.b = fr.b; ff.y = fr.y;
        ff.lb = fr.lb; ff.ub = fr.ub; ff.Dinv = fr.Dinv; ff.Cw = fr.Cw;
        ff.d1 = fr.d1; ff.g = fr.g;
        ff.d2 = d2->d;
        ff.d1out = t1->d;
        ff.V = fr.V; ff.alpha = fr.alpha; ff.beta = fr.beta;
        ff.ncols = m; ff.accumulate = accumulate; ff.from_vars = fr.from_vars;
        ff.b0sig = fr.b0sig; ff.mu = fr.mu; ff.mu_rhs = fr.mu_rhs; ff.k = k;
        ff.cbank = -1;
        ff.apz = apz_w;
        ff.nca = ncon;
        rc = pcu_launch_wide<Pass2R1F<0, 1>, 1>(ctx, ff, nvars, wd, NO_RED, m);
        if (rc > 0) return 1;
        if (rc == 0) {
          apz_done(accumulate, apz_w);
          pass1_r.assign(m, 0.0);
          if (ctx->big_fetch(m, pass1_r.data())) return 1;
          std::swap(d1, t1);
          pass1_ready = 1;
        }
      }
      if (rc < 0) {
        fr.apz = apz_w;
        fr.nca = ncon;
        if (launch_tile(ctx, fr, nvars, wd, NO_RED)) return 1;
        apz_done(accumulate, fr.apz);
      }
    }
    denseResidual(vars, mu_res, b, &y, VTp);
    if (emitted) *emitted = 1;
    return 0;
  }
  if (stats_tau > 0.0 && !opt_no_fuse2s) {
    // last pass of the iteration's solves: take the step statistics on the way
    Pass2SF fs;
    fs.v = f2.v; fs.b = f2.b; fs.y = f2.y;
    fs.lb = f2.lb; fs.ub = f2.ub; fs.Dinv = f2.Dinv; fs.Cw = f2.Cw;
    fs.d1 = f2.d1; fs.d2 = f2.d2; fs.g = g->d;
    fs.V = f2.V; fs.alpha = f2.alpha; fs.ncols = f2.ncols;
    fs.accumulate = f2.accumulate; fs.tau = stats_tau; fs.k = f2.k;
    fs.cbank = -1;
    fs.apz = apz_target(accumulate, true);
    fs.nca = ncon;
    RedBuf rb = ctx->redbuf(Pass2SF::NS, Pass2SF::NX, Pass2SF::NM);
    int rcw = -1;
    if (m > 32 && !opt_no_wide) {
      rcw = pcu_launch_wide<Pass2SF, 0>(ctx, fs, nvars, wd, rb, m);
      if (rcw > 0) return 1;
    }
    if (rcw < 0 && launch_tile(ctx, fs, nvars, wd, rb)) return 1;
    apz_done(accumulate, fs.apz);
    if (ctx->fetch(stats_out)) return 1;
    stats_ready = 1;
    stats_tau_used = stats_tau;
  } else {
    apz_target(accumulate, false);
    if (launch_tile(ctx, f2, nvars, wd, NO_RED)) return 1;
  }
  if (VTp && !derived) {
    ColTable Vall;
    for (int j = 0; j < ncon; j++) Vall.p[j] = Ac[j]->d;
    if (qa > 0) qn->z_table(Vall, ncon);
    if (ncon + qa > 0) {
      if (pcu_mdot_enqueue(ctx, y.v[PCU_X]->d, Vall, ncon + qa, nvars, 0)) return 1;
      if (ctx->big_fetch(ncon + qa, VTp)) return 1;
    }
  }
  return 0;
}

// ------------------------------------------------------------------ kktChain
// The KKT solve of a default iteration (monotone barrier, one refinement step,
// ncon + q <= 32, right-hand side from the variables) as ONE stream-ordered chain:
//   DiagRhsF -> Gram (+ all-reduce) -> pcu_dense_solve -> Pass2SVF -> fetch.
// The iterative refinement is done in the column space of [A|Z] by the small dense
// algebra (pcu_dense.cuh: pcu_dense_solve), so one pass applies the refined step and
// takes its statistics.  on_device: the dense algebra runs in pcu_dense_kernel on a
// flat device buffer, the pass reads its coefficients from the constant bank, and the
// chain needs no host round trip; otherwise the same statements run on the host
// between the Gram result and the pass.  Same arithmetic as setUpKKTDiagRhs +
// setUpKKTSystem + computeKKTStep x 2 (IP.cpp:1832-1971, 2634-2737, 4971-4991) up to
// the rounding of the refinement residual's elementwise operations.
int pcu_dense_enqueue(cudaStream_t stream, double *buf, const DenseOff &o, const double *Sin);
void pcu_dense_host(double *w, const DenseOff &o, const double *Sin);

int pcu_ip::kktChain(Vars &vars, Vars &b, Vars &y, int use_qn, double mu, double tau,
                     double *VTp, int on_device) {
  const int q = (qn && use_qn) ? qn->size() : 0;
  const int m = ncon + q;
  if (m < 1 || m > PCU_DENSE_MAXM) return 1;
  stats_ready = 0;
  pass1_ready = 0;
  if (setUpKKTDiagRhs(vars, use_qn, mu)) return 1;
  // ---- inputs of the dense algebra (1-7 KB)
  const int ld = 8 * ((m + 1 + 7) / 8);
  const DenseOff o = pcu_dense_offsets(ncon, q, ld);
  if (denseReserve(o)) return 1;
  if (on_device && !dense_dev) PCU_CUDA_OK(cudaMalloc(&dense_dev, sizeof(double) * dense_cap));
  dense_off = o;
  double *h = dense_host;
  densePack(o, vars, mu, nullptr);
  if (on_device)
    PCU_CUDA_OK(cudaMemcpyAsync(dense_dev, h, sizeof(double) * o.S, cudaMemcpyHostToDevice,
                                ctx->stream));
  // ---- Gram pass with the first solve's right-hand side as column m
  ColTable V;
  for (int j = 0; j < ncon; j++) V.p[j] = Ac[j]->d;
  if (q > 0) qn->z_table(V, ncon);
  ColTable Vg = V;
  Vg.p[m] = d1->d;
  int ldg = 0;
  if (pcu_gram_enqueue(ctx, Vg, m + 1, Dinv->d, Cw->d, wd, nvars, &ldg, d2->d, m)) return 1;
  if (ldg != ld) return 1;
  // ---- the dense algebra, refinement included
  if (on_device) {
    if (ctx->world > 1) {
      NcclApi &api = nccl_api();
      if (api.AllReduce(ctx->d_big, ctx->d_big, (size_t)ld * ld, ncclFloat64, ncclSum,
                        ctx->comm, ctx->stream) != ncclSuccess)
        return 1;
    }
    ctx->prof_begin("dense_kernel");
    if (pcu_dense_enqueue(ctx->stream, dense_dev, o, ctx->d_big)) return 1;
    ctx->prof_end();
    ctx->launches++;
    // the pass's coefficients: device buffer -> constant bank, stream-ordered
    PCU_CUDA_OK(cudaMemcpyToSymbolAsync(pcu_chain_coef, dense_dev + o.coef,
                                        sizeof(double) * PCU_DENSE_MAXM, 0,
                                        cudaMemcpyDeviceToDevice, ctx->stream));
    // what the dense kernel produced (dense step, [A|Z]^T p, the factors) goes to the
    // host BEFORE the pass is enqueued: its reduction flag then implies the copy (the
    // fetch below polls that flag, it does not synchronise the stream)
    PCU_CUDA_OK(cudaMemcpyAsync(h + o.S, dense_dev + o.S, sizeof(double) * (o.total - o.S),
                                cudaMemcpyDeviceToHost, ctx->stream));
  } else {
    std::vector<double> Sg((size_t)ld * ld);
    if (ctx->big_fetch((size_t)ld * ld, Sg.data())) return 1;
    pcu_dense_host(h, o, Sg.data());
  }
  // ---- the one pass: the refined step + the step statistics
  auto pass = [&](auto fs) -> int {
    fs.v = vars.dv(); fs.b = b.dv(); fs.y = y.dv();
    fs.lb = lb->d; fs.ub = ub->d; fs.Dinv = Dinv->d; fs.Cw = Cw->d;
    fs.d1 = d1->d; fs.d2 = d2->d; fs.g = g->d;
    fs.V = V;
    fs.cbank = on_device ? 0 : -1;
    if (!on_device)
      for (int j = 0; j < m; j++) fs.alpha.v[j] = h[o.coef + j];
    fs.ncols = m;
    fs.accumulate = 0; fs.tau = tau; fs.mu_rhs = mu; fs.k = kconst();
    fs.apz = apz_target(0, true);
    fs.nca = ncon;
    typedef decltype(fs) F;
    RedBuf rb = ctx->redbuf(F::NS, F::NX, F::NM);
    if (launch_tile(ctx, fs, nvars, wd, rb)) return 1;
    apz_done(0, fs.apz);
    PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k1, ctx->stream));
    return ctx->fetch(stats_out);
  };
  if (opt.use_diag_hessian) {
    Pass2SVHF fs;
    fs.h = hdiag->d;
    if (pass(fs)) return 1;
    // sum h p^2 follows the 22 sums of StatsF's layout: take it out, so that the maximum
    // and the minima sit where stepStats reads them
    const int ns = StatsF::NS;
    stats_hp2 = stats_out[ns];
    for (int i = ns; i < ns + StatsF::NX + StatsF::NM; i++) stats_out[i] = stats_out[i + 1];
  } else if (pass(Pass2SVF())) {
    return 1;
  }
  stats_ready = 1;
  stats_tau_used = tau;
  // ---- host mirrors of what the dense algebra produced
  for (int i = 0; i < ncon; i++) {
    y.z[i] = h[o.yz + i];
    y.s[i] = h[o.ys + i];
    y.t[i] = h[o.yt + i];
    y.zs[i] = h[o.yzs + i];
    y.zt[i] = h[o.yzt + i];
    b.z[i] = h[o.bz + i];
    b.s[i] = h[o.bs + i];
    b.t[i] = h[o.bt + i];
    b.zs[i] = h[o.bzs + i];
    b.zt[i] = h[o.bzt + i];
  }
  for (int i = 0; i < m; i++) VTp[i] = h[o.vtp + i];
  return 0;
}

// addMehrotraCorrectorResidual (IP.cpp:1729-1789)
int pcu_ip::addMehrotraCorrectorResidual(Vars &step, Vars &res) {
  for (int i = 0; i < ncon; i++) {
    res.zs[i] -= step.s[i] * step.zs[i];
    res.zt[i] -= step.t[i] * step.zt[i];
  }
  MehrotraCorrF f;
  f.p = step.dv();
  f.r = res.dv();
  f.lb = lb->d;
  f.ub = ub->d;
  f.k = kconst();
  return launch_tile(ctx, f, nvars, wd, NO_RED);
}

int pcu_ip::stepStats(Vars &vars, Vars &step, double tau, double *sums,
                      double *mins) {
  double out[StatsF::NS + StatsF::NX + StatsF::NM];
  if (stats_ready && stats_tau_used == tau) {
    // taken by the last pass of the KKT solve (Pass2SF)
    memcpy(out, stats_out, sizeof(out));
    stats_ready = 0;
  } else {
    StatsF f;
    f.v = vars.dv();
    f.p = step.dv();
    f.lb = lb->d;
    f.ub = ub->d;
    f.g = g->d;
    f.tau = tau;
    f.k = kconst();
    RedBuf rb = ctx->redbuf(StatsF::NS, StatsF::NX, StatsF::NM);
    if (launch_tile(ctx, f, nvars, wd, rb)) return 1;
    if (ctx->fetch(out)) return 1;
  }
  memcpy(sums, out, sizeof(double) * StatsF::NS);
  stats_pmax = out[StatsF::NS];
  mins[0] = std::min(1.0, out[StatsF::NS + 1]);
  mins[1] = std::min(1.0, out[StatsF::NS + 2]);
  // dense slack / multiplier steps (IP.cpp:2986-3017)
  for (int i = 0; i < ncon; i++) {
    if (step.s[i] < 0.0) mins[0] = std::min(mins[0], -tau * vars.s[i] / step.s[i]);
    if (step.t[i] < 0.0) mins[0] = std::min(mins[0], -tau * vars.t[i] / step.t[i]);
    if (step.zs[i] < 0.0) mins[1] = std::min(mins[1], -tau * vars.zs[i] / step.zs[i]);
    if (step.zt[i] < 0.0) mins[1] = std::min(mins[1], -tau * vars.zt[i] / step.zt[i]);
  }
  return 0;
}

// ---------------------------------------------- initLeastSquaresMultipliers
// IP.cpp:5366-5534
struct MaskBoundMultF : NoStreams {  // zl = 0 where lb <= -mbv, zu = 0 where ub >= mbv
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *lb, *ub;
  double *zl, *zu;
  double mbv;
  // affine start (IP.cpp:5629-5651): z = max(mn, |z + pz|) where the bound exists
  const double *pzl, *pzu;
  double mn;
  int affine;
  // least-squares right-hand side rx = -(g - zl + zu) (IP.cpp:5472-5475)
  const double *g;
  double *rx;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
    double l[W], u[W], a[W], b[W];
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(zl, i, a);
    ldv<W>(zu, i, b);
    if (affine) {
      double pa[W], pb[W];
      ldv<W>(pzl, i, pa);
      ldv<W>(pzu, i, pb);
#pragma unroll
      for (int e = 0; e < W; e++) {
        if (l[e] > -mbv) a[e] = fmax(mn, fabs(a[e] + pa[e]));
        if (u[e] < mbv) b[e] = fmax(mn, fabs(b[e] + pb[e]));
      }
    }
#pragma unroll
    for (int e = 0; e < W; e++) {
      if (l[e] <= -mbv) a[e] = 0.0;
      if (u[e] >= mbv) b[e] = 0.0;
    }
    stv<W>(zl, i, a);
    stv<W>(zu, i, b);
    if (rx) {
      double gv[W], r[W];
      ldv<W>(g, i, gv);
#pragma unroll
      for (int e = 0; e < W; e++) r[e] = -((gv[e] - a[e]) + b[e]);
      stv<W>(rx, i, r);
    }
  }
};

struct SparseStartF : NoStreams {  // W-sized pieces of the starting-point strategies
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  DVars v, p;
  double mn, gamma;
  int nwineq;
  int mode;  // 0: clip zw to +-10 gamma (IP.cpp:5520-5533); 1: affine (IP.cpp:5605-5627)
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
      const long long ci = i + e;
      if (mode == 0) {
        const double gam = 10.0 * gamma;  // max(gamma_sw, gamma_tw) = gamma
        const double zw = v.zw[ci];
        if (zw < -gam || zw > gam) v.zw[ci] = 0.0;
      } else {
        v.zw[ci] = v.zw[ci] + p.zw[ci];
        v.sw[ci] = fmax(mn, fabs(v.sw[ci] + p.sw[ci]));
        v.tw[ci] = fmax(mn, fabs(v.tw[ci] + p.tw[ci]));
        v.zsw[ci] = fmax(mn, fabs(v.zsw[ci] + p.zsw[ci]));
        v.ztw[ci] = fmax(mn, fabs(v.ztw[ci] + p.ztw[ci]));
      }
    }
  }
};

int pcu_ip::initLeastSquaresMultipliers() {
  Vars &vars = variables, &res = residual;
  const double mu0 = opt.init_barrier_param;
  for (int i = 1; i < 8; i++)
    if (pcu_vec_set(vars.v[i], mu0)) return 1;
  for (int i = 0; i < ncon; i++)
    vars.z[i] = vars.s[i] = vars.t[i] = vars.zs[i] = vars.zt[i] = mu0;
  WDesc w0;
  memset(&w0, 0, sizeof(w0));
  // zero out-of-range bound multipliers and form rx = -(g - zl + zu)
  MaskBoundMultF fm;
  fm.lb = lb->d;
  fm.ub = ub->d;
  fm.zl = vars.v[PCU_ZL]->d;
  fm.zu = vars.v[PCU_ZU]->d;
  fm.mbv = opt.max_bound_value;
  fm.affine = 0;
  fm.pzl = fm.pzu = nullptr;
  fm.mn = 0.0;
  fm.g = g->d;
  fm.rx = res.v[PCU_X]->d;
  if (launch_tile(ctx, fm, nvars, w0, NO_RED)) return 1;
  // D = I, C = small (IP.cpp:5418-5431), G = small*I + A^T D0^-1 A
  if (setUpKKTDiagSystem(vars, 0, 1)) return 1;
  std::vector<double> small(ncon, 1e-4);
  if (setUpKKTSystem(vars, 0, small.data())) return 1;
  // Right-hand side: only bx is non-zero.  With b.zl = b.zu = 0 and zero
  // sparse/dense parts the full solve reduces to IP.cpp:5478-5508.
  for (int i = 1; i < 8; i++)
    if (pcu_vec_zero(res.v[i])) return 1;
  for (int i = 0; i < ncon; i++) res.z[i] = res.s[i] = res.t[i] = res.zs[i] = res.zt[i] = 0.0;
  // The dense solve of the reference here is z = -G^-1 A^T yx with no slack
  // terms: emulate with s = t = 0 contributions by calling the generic step with
  // temporary unit slacks (b dense parts are zero so only G matters).
  Vars &step = update;
  // Use the low-level pieces directly: pass 1, mdot, solve, pass 2.
  {
    Pass1F f1;
    f1.v = vars.dv();
    f1.b = res.dv();
    f1.lb = lb->d;
    f1.ub = ub->d;
    f1.Dinv = Dinv->d;
    f1.Cw = Cw->d;
    f1.d1 = d1->d;
    f1.d2 = d2->d;
    f1.t1 = t1->d;
    f1.k = kconst();
    if (launch_tile(ctx, f1, nvars, wd, NO_RED)) return 1;
    ColTable V;
    for (int j = 0; j < ncon; j++) V.p[j] = Ac[j]->d;
    std::vector<double> z(ncon);
    if (ncon > 0) {
      if (pcu_mdot_enqueue(ctx, t1->d, V, ncon, nvars, 0)) return 1;
      if (ctx->big_fetch(ncon, z.data())) return 1;
      for (int i = 0; i < ncon; i++) z[i] = -z[i];
      const double *h = dense_host;
      const DenseOff &o = dense_off;
      pcu_dense_lu_solve(ncon, h + o.Gfac, h + o.gpiv, h + o.ginv, z.data());
    }
    Pass2F f2;
    for (int i = 0; i < ncon; i++) f2.alpha.v[i] = z[i];
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
    f2.k = kconst();
    if (launch_tile(ctx, f2, nvars, wd, NO_RED)) return 1;
    // vars.z = z, vars.zw = yw (IP.cpp:5483-5508)
    for (int i = 0; i < ncon; i++) {
      const double gam = 10.0 * std::max(gamma_s[i], gamma_t[i]);
      vars.z[i] = (z[i] < -gam || z[i] > gam) ? 0.0 : z[i];
    }
    if (pcu_vec_copy(vars.v[PCU_ZW], step.v[PCU_ZW])) return 1;
  }
  if (nwcon > 0) {
    SparseStartF fs;
    fs.v = vars.dv();
    fs.p = step.dv();
    fs.mn = 0.0;
    fs.gamma = opt.penalty_gamma;
    fs.nwineq = prob->nwinequality;
    fs.mode = 0;
    if (launch_tile(ctx, fs, nwcon, w0, NO_RED)) return 1;
  }
  return 0;
}

// ------------------------------------------------ initAffineStepMultipliers
// IP.cpp:5536-5656
int pcu_ip::initAffineStepMultipliers() {
  Vars &vars = variables, &res = residual, &step = update;
  if (initLeastSquaresMultipliers()) return 1;
  // (out-of-range multipliers are already zero)
  if (computeKKTRes(vars, 0.0, res, nullptr, nullptr, nullptr)) return 1;
  // (the GMRES preconditioner switch also acts here, IP.cpp:5575-5578)
  int use_qn = (opt.sequential_linear_method || !opt.use_qn_gmres_precon) ? 0 : 1;
  if (setUpKKTDiagSystem(vars, use_qn, 0)) return 1;
  if (setUpKKTSystem(vars, use_qn, nullptr)) return 1;
  if (computeKKTStep(vars, res, step, use_qn, 0, nullptr, 0, 0.0, nullptr)) return 1;
  const double mn = opt.start_affine_multiplier_min;
  for (int i = 0; i < ncon; i++) {
    vars.z[i] = vars.z[i] + step.z[i];
    vars.s[i] = std::max(mn, fabs(vars.s[i] + step.s[i]));
    vars.t[i] = std::max(mn, fabs(vars.t[i] + step.t[i]));
    vars.zs[i] = std::max(mn, fabs(vars.zs[i] + step.zs[i]));
    vars.zt[i] = std::max(mn, fabs(vars.zt[i] + step.zt[i]));
  }
  WDesc w0;
  memset(&w0, 0, sizeof(w0));
  if (nwcon > 0) {
    SparseStartF fs;
    fs.v = vars.dv();
    fs.p = step.dv();
    fs.mn = mn;
    fs.gamma = opt.penalty_gamma;
    fs.nwineq = prob->nwinequality;
    fs.mode = 1;
    if (launch_tile(ctx, fs, nwcon, w0, NO_RED)) return 1;
  }
  MaskBoundMultF fm;
  fm.lb = lb->d;
  fm.ub = ub->d;
  fm.zl = vars.v[PCU_ZL]->d;
  fm.zu = vars.v[PCU_ZU]->d;
  fm.mbv = opt.max_bound_value;
  fm.affine = 1;
  fm.pzl = step.v[PCU_ZL]->d;
  fm.pzu = step.v[PCU_ZU]->d;
  fm.mn = mn;
  fm.g = nullptr;
  fm.rx = nullptr;
  if (launch_tile(ctx, fm, nvars, w0, NO_RED)) return 1;
  // barrier_param = computeComp(vars) (IP.cpp:5655): statistics of a residual pass
  if (computeKKTRes(vars, 0.0, res, nullptr, nullptr, nullptr)) return 1;
  barrier_param = compFromStats(vars);
  return 0;
}

// ------------------------------------------------------------------ history
struct StateSumF : NoStreams {  // checksums of the iterate for the parity history
  static constexpr int NS = 7, NX = 1, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  DVars v;
  const double *g;
  int sparse;  // 0: N-sized pass, 1: W-sized pass
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
    if (!sparse) {
      double x[W], a[W], b[W], gv[W];
      ldv<W>(v.x, i, x);
      ldv<W>(v.zl, i, a);
      ldv<W>(v.zu, i, b);
      ldv<W>(g, i, gv);
#pragma unroll
      for (int e = 0; e < W; e++) {
        acc.s[0] += x[e];
        acc.s[1] = fma(x[e], x[e], acc.s[1]);
        acc.s[2] += a[e];
        acc.s[3] += b[e];
        acc.x[0] = fmax(acc.x[0], fabs(gv[e]));
      }
    } else {
      double a[W], b[W], c[W];
      ldv<W>(v.zw, i, a);
      ldv<W>(v.sw, i, b);
      ldv<W>(v.tw, i, c);
#pragma unroll
      for (int e = 0; e < W; e++) {
        acc.s[4] += a[e];
        acc.s[5] += b[e];
        acc.s[6] += c[e];
      }
    }
  }
};

int pcu_ip::snapshot(int k, double comp, double max_prime, double max_dual,
                     double max_infeas, double res_norm) {
  if (opt.history_level <= 0) return 0;
  HistRec rec;
  memset(rec.f, 0, sizeof(rec.f));
  double sums[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (opt.history_level >= 2) {
    WDesc w0;
    memset(&w0, 0, sizeof(w0));
    StateSumF f;
    f.v = variables.dv();
    f.g = g->d;
    f.sparse = 0;
    RedBuf rb = ctx->redbuf(7, 1, 0);
    if (launch_tile(ctx, f, nvars, w0, rb)) return 1;
    double o1[8], o2[8];
    if (ctx->fetch(o1)) return 1;
    memcpy(sums, o1, sizeof(o1));
    if (nwcon > 0 || ctx->world > 1) {
      f.sparse = 1;
      RedBuf rb2 = ctx->redbuf(7, 1, 0);
      if (launch_tile(ctx, f, nwcon, w0, rb2)) return 1;
      if (ctx->fetch(o2)) return 1;
      sums[4] = o2[4];
      sums[5] = o2[5];
      sums[6] = o2[6];
    }
  }
  double *f = rec.f;
  f[0] = k;
  f[1] = fobj;
  f[2] = barrier_param;
  f[3] = rho_penalty_search;
  f[4] = comp;
  f[5] = max_prime;
  f[6] = max_dual;
  f[7] = max_infeas;
  f[8] = res_norm;
  f[9] = neval;
  f[10] = ngeval;
  f[11] = ls.alpha_prev;
  f[12] = ls.last_pnorm2;
  f[13] = qn ? qn->b0 : 0.0;
  f[14] = qn ? qn->size() : 0;
  f[15] = sums[0];
  f[16] = sqrt(sums[1]);
  f[17] = sums[2];
  f[18] = sums[3];
  f[19] = sums[4];
  f[20] = sums[5];
  f[21] = sums[6];
  f[22] = sums[7];
  f[23] = ls.alpha_xprev;
  f[24] = ls.alpha_zprev;
  f[25] = nhvec;
  rec.dense.reserve(6 * ncon);
  const std::vector<double> *parts[6] = {&c, &variables.z, &variables.s,
                                         &variables.t, &variables.zs,
                                         &variables.zt};
  for (auto p : parts) rec.dense.insert(rec.dense.end(), p->begin(), p->end());
  rec.info = ls.info;
  history.push_back(rec);
  return 0;
}

// Text log row, same format as the reference (IP.cpp:4777-4801)
void pcu_ip::log_line(int k, double comp, double max_prime, double max_infeas,
                      double max_dual) {
  if (!outfp || ctx->rank != 0) return;
  if (k % 10 == 0 || opt.output_level > 0) {
    fprintf(outfp,
            "\n%4s %4s %4s %4s %7s %7s %7s %12s %7s %7s %7s %7s %7s %8s %7s info\n",
            "iter", "nobj", "ngrd", "nhvc", "alpha", "alphx", "alphz", "fobj",
            "|opt|", "|infes|", "|dual|", "mu", "comp", "dmerit", "rho");
  }
  if (k == 0) {
    fprintf(outfp,
            "%4d %4d %4d %4d %7s %7s %7s %12.5e %7.1e %7.1e %7.1e %7.1e %7.1e %8s %7s %s\n",
            k, neval, ngeval, nhvec, "--", "--", "--", fobj, max_prime, max_infeas,
            max_dual, barrier_param, comp, "--", "--", ls.info.c_str());
  } else {
    fprintf(outfp,
            "%4d %4d %4d %4d %7.1e %7.1e %7.1e %12.5e %7.1e %7.1e %7.1e %7.1e %7.1e %8.1e %7.1e %s\n",
            k, neval, ngeval, nhvec, ls.alpha_prev, ls.alpha_xprev, ls.alpha_zprev,
            fobj, max_prime, max_infeas, max_dual, barrier_param, comp,
            ls.dm0_prev, rho_penalty_search, ls.info.c_str());
  }
  fflush(outfp);
}

// scaleKKTStep (IP.cpp:3196-3274) + evalMeritInitDeriv (IP.cpp:3652-3924) from
// ONE statistics pass; the step itself stays unscaled on the device.
// fixed_scale < 0: the step lengths come from the fraction-to-boundary rule and
// the step is treated as scaled by alpha_x (the optimizer's path).
// fixed_scale >= 0: the step is taken as already scaled (factor 1) and
// fixed_scale is the max_x argument of the reference's evalMeritInitDeriv.
int pcu_ip::scaleAndMerit(Vars &v, Vars &upd, double tau, double comp,
                          const double *VTp, double fixed_scale,
                          StepScale *out, int inexact_newton_step) {
  const double abs_res_tol = opt.abs_res_tol;
  const int slm = opt.sequential_linear_method;
  const int nA = ncon;
  double sums[StatsF::NS], mins[2];
  double alpha_x = 1.0, alpha_z = 1.0, m0 = 0.0, dm0 = 0.0, pnorm2 = 0.0;
  int ceq_step = 0;
    // (stepStats consumes the statistics of the pass that formed the step)
    const bool hp2_ready = stats_ready && stats_tau_used == tau;
    const double hp2 = stats_hp2;
    if (stepStats(v, upd, tau, sums, mins)) return 1;
    alpha_x = mins[0];
    alpha_z = mins[1];
    ceq_step = 0;
    const double max_bnd = 100.0;
    if (alpha_x > alpha_z) {
      if (alpha_x > max_bnd * alpha_z) alpha_x = max_bnd * alpha_z;
      else if (alpha_x < alpha_z / max_bnd) alpha_x = alpha_z / max_bnd;
    } else {
      if (alpha_z > max_bnd * alpha_x) alpha_z = max_bnd * alpha_x;
      else if (alpha_z < alpha_x / max_bnd) alpha_z = alpha_x / max_bnd;
    }
    double product = (sums[0] + alpha_x * sums[1] + alpha_z * sums[2] +
                      alpha_x * alpha_z * sums[3]) / opt.rel_bound_barrier +
                     (sums[4] + alpha_x * sums[5] + alpha_z * sums[6] +
                      alpha_x * alpha_z * sums[7]);
    double count = res_sums[1];
    for (int i = 0; i < ncon; i++) {
      product += (v.s[i] + alpha_x * upd.s[i]) * (v.zs[i] + alpha_z * upd.zs[i]) +
                 (v.t[i] + alpha_x * upd.t[i]) * (v.zt[i] + alpha_z * upd.zt[i]);
      count += 2.0;
    }
    const double comp_new = count != 0.0 ? product / count : 0.0;
    if (comp_new > 10.0 * comp) {
      ceq_step = 1;
      if (alpha_x > alpha_z) alpha_x = alpha_z;
      else alpha_z = alpha_x;
    }
    if (inexact_newton_step) {  // IP.cpp:3241-3248: one step length, no other rule
      alpha_x = alpha_z = std::min(mins[0], mins[1]);
      ceq_step = 0;
    }
    if (fixed_scale >= 0.0) {
      alpha_x = 1.0;
      alpha_z = 1.0;
      ceq_step = 0;
    }
    pnorm2 = alpha_x * alpha_x * sums[17];
    // ---- merit function and derivative with the step scaled by alpha_x ----
    const double kap = opt.rel_bound_barrier;
    double pos = sums[8] * kap + sums[12], neg = sums[9] * kap + sums[13];
    double ppos = alpha_x * (sums[10] * kap + sums[14]);
    double pneg = alpha_x * (sums[11] * kap + sums[15]);
    for (int i = 0; i < ncon; i++) {
      const double lsv = log(v.s[i]), ltv = log(v.t[i]);
      if (v.s[i] > 1.0) pos += lsv; else neg += lsv;
      if (v.t[i] > 1.0) pos += ltv; else neg += ltv;
      const double ps = alpha_x * upd.s[i], pt = alpha_x * upd.t[i];
      if (ps > 0.0) ppos += ps / v.s[i]; else pneg += ps / v.s[i];
      if (pt > 0.0) ppos += pt / v.t[i]; else pneg += pt / v.t[i];
    }
    // evalInfeasDeriv (IP.cpp:3465-3509)
    double dense_infeas = 0.0, pdense_infeas = 0.0;
    for (int i = 0; i < ncon; i++) {
      const double cval = c[i] - v.s[i] + v.t[i];
      const double pcval = alpha_x * (VTp[i] - upd.s[i] + upd.t[i]);
      dense_infeas += cval * cval;
      pdense_infeas += cval * pcval;
    }
    const double infeas = sqrt(dense_infeas + sums[20]);
    const double psparse = alpha_x * sums[21];
    const double infeas_proj = infeas > 0.0 ? (pdense_infeas + psparse) / infeas : 0.0;
    // p^T B p through the compact form (IP.cpp:3820-3821)
    double pTBp = 0.0;
    if (opt.use_diag_hessian) {
      // the compact form's expression with B = diag(h): sum h p^2, taken by the pass that
      // formed the step (Pass2SVHF); a step from elsewhere has no such sum
      if (!hp2_ready) {
        fprintf(stderr, "ParOpt error: use_diag_hessian: this step has no p^T diag(h) p\n");
        return 1;
      }
      pTBp = 0.5 * alpha_x * alpha_x * hp2;
    } else if (qn && !slm) {
      double v2 = qn->b0 * sums[17];
      const int q = qn->size();
      if (q > 0) {
        std::vector<double> kapq(q);
        qn->solve_compact(VTp + nA, kapq.data());
        for (int i = 0; i < q; i++) v2 -= kapq[i] * VTp[nA + i];
      }
      pTBp = 0.5 * alpha_x * alpha_x * v2;
    }
    double merit = fobj + sums[18] - barrier_param * (pos + neg);
    double pmerit = alpha_x * sums[16] + alpha_x * sums[19] -
                    barrier_param * (ppos + pneg);
    for (int i = 0; i < ncon; i++) {
      merit += gamma_s[i] * v.s[i] + gamma_t[i] * v.t[i];
      pmerit += alpha_x * (gamma_s[i] * upd.s[i] + gamma_t[i] * upd.t[i]);
    }
    double numer = pmerit;
    if (pTBp > 0.0) numer += 0.5 * pTBp;
    const double pdf = opt.penalty_descent_fraction;
    const double max_x = fixed_scale >= 0.0 ? fixed_scale : alpha_x;
    double rho_hat = 0.0;
    if (infeas < 0.1 * abs_res_tol) {
      const double denom = -(1.0 - pdf) * max_x * infeas;
      if (numer >= 0.0 && denom < 0.0) rho_hat = -numer / denom;
    } else {
      double denom = infeas_proj + pdf * max_x * infeas;
      if (numer >= 0.0) {
        if (denom < 0.0) {
          rho_hat = -numer / denom;
        } else {
          denom = -(1.0 - pdf) * max_x * infeas;
          rho_hat = -numer / denom;
        }
      }
    }
    if (rho_hat > rho_penalty_search) {
      rho_penalty_search = rho_hat;
    } else {
      rho_penalty_search *= 0.5;
      if (rho_penalty_search < rho_hat) rho_penalty_search = rho_hat;
    }
    if (rho_penalty_search < opt.min_rho_penalty_search)
      rho_penalty_search = opt.min_rho_penalty_search;
    merit += rho_penalty_search * infeas;
    if (infeas < 0.1 * abs_res_tol) pmerit -= rho_penalty_search * max_x * infeas;
    else pmerit += rho_penalty_search * infeas_proj;
    m0 = merit;
    dm0 = pmerit;
    out->alpha_x = alpha_x;
    out->alpha_z = alpha_z;
    out->ceq = ceq_step;
    out->m0 = m0;
    out->dm0 = dm0;
    out->pnorm2 = pnorm2;
    return 0;
}

// --------------------------------------------------------- use_diag_hessian
// The diagonal Hessian runs on the default iteration's route only: monotone barrier,
// one refinement step done in the column space of [A|Z] (kktChain) with 1 <= ncon <= 32
// dense constraints, any starting-point strategy.  Everything else is refused here
// rather than run with a Hessian term missing.
int pcu_ip::diagHessianRefused() {
  if (!opt.use_diag_hessian) return 0;
  const char *why = nullptr;
  if (!prob->hasHessianDiag()) why = "the problem has no evalHessianDiag";
  else if (opt.use_hvec_product) why = "use_hvec_product is not available with it";
  else if (qn_external) why = "a quasi-Newton object set by setQuasiNewton is not used with it";
  else if (opt.sequential_linear_method) why = "sequential_linear_method is not available with it";
  else if (opt.barrier_strategy != "monotone") why = "it needs barrier_strategy = monotone";
  else if (opt.iterative_refinement_steps != 1) why = "it needs iterative_refinement_steps = 1";
  else if (ncon < 1 || ncon > 32) why = "it needs 1 to 32 dense constraints";
  if (why) {
    if (ctx->rank == 0) fprintf(stderr, "ParOpt error: use_diag_hessian: %s\n", why);
    return 1;
  }
  if (!hdiag) hdiag = pcu_vec_create(ctx, nvars);
  return hdiag ? 0 : 1;
}

// -------------------------------------------------------------------- begin
// Everything ParOptInteriorPoint::optimize does before its major loop
// (IP.cpp:4399-4606).
int pcu_ip::begin() {
  gaz_valid = 0;
  apz_state = 0;
  if (diagHessianRefused()) return 1;
  if (ensure_qn()) return 1;
  refresh_penalties();
  if (!opt.output_file.empty() && !outfp && ctx->rank == 0) {
    outfp = fopen(opt.output_file.c_str(), "w");
  }
  ls = LoopState();
  auto strat = [](const std::string &s) {
    if (s == "monotone") return (int)BS_MONOTONE;
    if (s == "mehrotra") return (int)BS_MEHROTRA;
    if (s == "mehrotra_predictor_corrector") return (int)BS_MPC;
    return (int)BS_COMP_FRACTION;
  };
  ls.barrier_strategy = BS_MONOTONE;
  ls.input_barrier_strategy = strat(opt.barrier_strategy);
  barrier_param = opt.init_barrier_param;
  rho_penalty_search = opt.init_rho_penalty_search;
  niter = neval = ngeval = nhvec = 0;
  status = 0;
  history.clear();
  times.clear();
  if (!opt.sequential_linear_method && !qn && !opt.use_diag_hessian) {
    if (ctx->rank == 0)
      fprintf(stderr,
              "ParOpt Error: Must use a sequential linear method if no "
              "quasi-Newton approximation is defined\n");
    return 1;
  }
  if (initAndCheckDesignAndBounds()) return 1;
  if (evalObjCon(variables.v[PCU_X])) {
    fprintf(stderr, "ParOpt: Initial function and constraint evaluation failed\n");
    return 1;
  }
  if (evalObjConGradient(variables.v[PCU_X], 1)) {
    fprintf(stderr, "ParOpt: Initial gradient evaluation failed\n");
    return 1;
  }
  if (opt.starting_point_strategy == "affine_step") {
    if (initAffineStepMultipliers()) return 1;
  } else if (opt.starting_point_strategy == "least_squares_multipliers") {
    if (initLeastSquaresMultipliers()) return 1;
  }
  if (pcu_ctx_sync(ctx)) return 1;
  cb_collect();
  ls.started = 1;
  return 0;
}

// ------------------------------------------------------------- iterate_once
// One pass of the major loop body (IP.cpp:4607-5329).
int pcu_ip::iterate_once(int *converged) {
  *converged = 0;
  if (!ls.started || ls.finished) return ls.finished ? 0 : 1;
  Vars &v = variables, &res = residual, &upd = update, &ref = refine;
  const int k = ls.k;
  const double abs_res_tol = opt.abs_res_tol;
  const double fp = opt.function_precision;
  const int uq = opt.use_quasi_newton_update;
  const int slm = opt.sequential_linear_method;
  // this iteration records into the other event set; the previous iteration's set is
  // read out below, once the first reduction of this iteration has synchronised
  ev_cur ^= 1;
  if (collect_times(evs[ev_cur])) return 1;  // (two iterations old: long finished)
  PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].it0, ctx->stream));
  // k0 / k1 bracket the KKT solve; give them a defined value for iterations that end early
  PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k0, ctx->stream));
  PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k1, ctx->stream));

  // (use_diag_hessian: diag(h) stands where the quasi-Newton object does; its "reset"
  // changes nothing, h comes from the problem, and is reported as the object's is)
  const bool hess_obj = qn || opt.use_diag_hessian;
  int qn_hessian_reset = 0;
  if (hess_obj && !slm) {
    if (k > 0 && k % opt.hessian_reset_freq == 0 && uq) {
      if (qn) qn->reset();
      qn_hessian_reset = 1;
    }
  }
  // the problem's writeOutput hook (IP.cpp:4620-4631)
  if (opt.write_output_frequency > 0 && k % opt.write_output_frequency == 0) {
    if (!opt.ip_checkpoint_file.empty() && !checkpoint_failed) {
      // a failed write is reported once and not tried again (IP.cpp:4622-4628)
      if (pcu_ip_write_solution(this, opt.ip_checkpoint_file.c_str())) {
        fprintf(stderr, "ParOpt: Checkpoint file %s creation failed\n",
                opt.ip_checkpoint_file.c_str());
        checkpoint_failed = 1;
      }
    }
    if (prob->writeOutput(k, v.v[PCU_X])) return 1;
  }
  const int rel_function_test =
      (ls.alpha_xprev == 1.0 && ls.alpha_zprev == 1.0 &&
       fabs(fobj - ls.fobj_prev) < opt.rel_func_tol * fabs(ls.fobj_prev));
  if (ls.no_merit_function_improvement) ls.line_search_test += 1;
  else ls.line_search_test = 0;

  double max_prime = 0.0, max_dual = 0.0, max_infeas = 0.0, res_norm = 0.0;
  int monotone_barrier_converged = 0;
  // monotone strategy with refinement: the residual vectors are never stored
  // (the GMRES right-hand side is the stored residual: no lazy residual with
  // use_hvec_product)
  const bool lazy_res = (ls.barrier_strategy == BS_MONOTONE) &&
                        opt.iterative_refinement_steps > 0 && !opt.use_hvec_product;
  // residual + norms + complementarity in one pass (IP.cpp:4656-4671)
  if (ls.barrier_strategy == BS_COMP_FRACTION) {
    // mu depends on comp: a first pass for comp, then the residual
    if (computeKKTRes(v, barrier_param, res, nullptr, nullptr, nullptr)) return 1;
  }
  double comp;
  if (ls.barrier_strategy == BS_COMP_FRACTION) {
    comp = compFromStats(v);
    // the history row shows the norms at the barrier the iteration starts with
    computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
    if (snapshot(k, comp, max_prime, max_dual, max_infeas, res_norm)) return 1;
    barrier_param = opt.monotone_barrier_fraction * comp;
    if (barrier_param < 0.1 * abs_res_tol) barrier_param = 0.1 * abs_res_tol;
    if (computeKKTRes(v, barrier_param, res, nullptr, nullptr, nullptr)) return 1;
    computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
    if (k == 0) ls.res_norm_prev = res_norm;
  } else {
    if (lazy_res && upd_stats_valid && norm_type_id() == 0) {
      // taken at this very point by the update passes of the previous iteration
      memcpy(res_sums, upd_sums, sizeof(res_sums));
      memcpy(res_max, upd_max, sizeof(res_max));
      memcpy(res_min, upd_min, sizeof(res_min));
      res_mu = barrier_param;
      res_has_step = 0;
      denseResidual(v, barrier_param, res, nullptr, nullptr);
    } else if (computeKKTRes(v, barrier_param, res, nullptr, nullptr, nullptr, lazy_res ? 0 : 1)) {
      // statistics only (lazy_res): the first solve recomputes the residual on the fly
      return 1;
    }
    upd_stats_valid = 0;
    comp = compFromStats(v);
    computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
    if (snapshot(k, comp, max_prime, max_dual, max_infeas, res_norm)) return 1;
    if (k == 0) ls.res_norm_prev = res_norm;
    if (ls.barrier_strategy == BS_MONOTONE) {
      if (k > 0 && ((res_norm < 10.0 * barrier_param) || rel_function_test ||
                    (ls.line_search_test >= 2))) {
        monotone_barrier_converged = 1;
      }
      if (monotone_barrier_converged) {  // IP.cpp:4695-4735
        if (barrier_param > 0.1 * abs_res_tol) ls.line_search_test = 0;
        const double mu_frac = opt.monotone_barrier_fraction * barrier_param;
        const double mu_pow = pow(barrier_param, opt.monotone_barrier_power);
        double new_mu = mu_frac;
        if (mu_pow < mu_frac) new_mu = mu_pow;
        if (new_mu < 0.1 * abs_res_tol) new_mu = 0.09999 * abs_res_tol;
        if (!(lazy_res && resNormAtBarrier(v, new_mu, res, &max_prime, &max_dual,
                                           &max_infeas, &res_norm))) {
          if (computeKKTRes(v, new_mu, res, nullptr, nullptr, nullptr, lazy_res ? 0 : 1))
            return 1;
          computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
        }
        rho_penalty_search = opt.min_rho_penalty_search;
        barrier_param = new_mu;
      }
    }
  }
  // the residual statistics above synchronised the stream: the previous iteration's
  // events are complete, reading them costs nothing
  if (collect_times(evs[ev_cur ^ 1])) return 1;
  last_comp = comp;
  log_line(k, comp, max_prime, max_infeas, max_dual);

  // convergence test (IP.cpp:4811-4840)
  if (k > 0 && (barrier_param <= 0.1 * abs_res_tol) &&
      (res_norm < abs_res_tol || rel_function_test || (ls.line_search_test >= 2))) {
    if (rel_function_test) status = 2;
    else if (ls.line_search_test >= 2) status = 3;
    else status = 1;
    if (outfp && ctx->rank == 0) {
      if (status == 2)
        fprintf(outfp, "\nParOpt: Successfully converged on relative function test\n");
      else if (status == 3)
        fprintf(outfp,
                "\nParOpt Warning: Current design point could not be improved. "
                "No barrier function decrease in previous two iterations\n");
      else
        fprintf(outfp, "\nParOpt: Successfully converged to requested tolerance\n");
      fflush(outfp);
    }
    ls.finished = 1;
    *converged = 1;
    return 0;
  }

  const int nA = ncon, nZ = qn ? qn->max_size() : 0;
  std::vector<double> VTp(nA + nZ + 1, 0.0);
  bool vtp_valid = true;

  // Newton or quasi-Newton step (IP.cpp:4842-4900): with exact Hessian-vector products
  // and small enough residuals, right-preconditioned GMRES on the exact KKT system
  int gmres_iters = 0, inexact_newton_step = 0;
  if (opt.use_hvec_product) {
    const double gmres_rtol = opt.eisenstat_walker_gamma *
                              pow(res_norm / ls.res_norm_prev, opt.eisenstat_walker_alpha);
    const double tol = opt.nk_switch_tol;
    if (max_prime < tol && max_dual < tol && max_infeas < tol &&
        gmres_rtol < opt.max_gmres_rtol) {
      const int use_qn_g = (slm || !opt.use_qn_gmres_precon) ? 0 : 1;
      PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k0, ctx->stream));
      if (setUpKKTDiagSystem(v, use_qn_g, 0)) return 1;
      if (setUpKKTSystem(v, use_qn_g, nullptr)) return 1;
      int err = 0;
      gmres_iters = computeKKTGMRESStep(v, res, upd, gmres_rtol, opt.gmres_atol, use_qn_g,
                                        VTp.data(), &err);
      if (err) return 1;
      PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k1, ctx->stream));
      if (gmres_iters < 0) {
        if (outfp && ctx->rank == 0 && opt.output_level > 0)
          fprintf(outfp, "      %9s\n", "step failed");
        // the residual was destroyed by the failed attempt (IP.cpp:4889-4893)
        if (computeKKTRes(v, barrier_param, res, nullptr, nullptr, nullptr)) return 1;
        computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
      } else {
        inexact_newton_step = 1;
      }
    }
  }

  ls.fobj_prev = fobj;
  ls.res_norm_prev = res_norm;
  int seq_linear_step = 0, diagonal_qn_step = 0;
  int use_qn = 1;
  if (inexact_newton_step) {
    // the step is there: none of the quasi-Newton step computations below run
  } else if (slm) {
    use_qn = 0;
  } else if (ls.line_search_failed && !uq) {
    use_qn = 0;
    seq_linear_step = 1;
    if (qn && qn->b0 > 0.0) {
      seq_linear_step = 0;
      diagonal_qn_step = 1;
    }
  }
  double mu_for_res = barrier_param;
  const bool mehrotra =
      ls.barrier_strategy == BS_MEHROTRA || ls.barrier_strategy == BS_MPC;
  if (mehrotra && !inexact_newton_step) {
    mu_for_res = 0.0;
    if (computeKKTRes(v, mu_for_res, res, nullptr, nullptr, nullptr)) return 1;
    computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
  }
  if (diagonal_qn_step) use_qn = 1;

  if (!inexact_newton_step) PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k0, ctx->stream));
  // The first solve's right-hand side can ride in the Gram pass when that solve
  // takes the fused residual-free route (see computeKKTStep).
  bool rhs_in_gram = false, wide_rhs = false;
  {
    const int qa = qn ? qn->size() : 0;
    const int q0 = (qn && use_qn) ? qa : 0;
    // (more than 32 columns: the wide Gram kernel takes the right-hand side as a plain
    // column, which needs a problem without weighting constraints)
    rhs_in_gram = lazy_res && !opt_no_rhsgram && !force_direct_dots &&
                  !diagonal_qn_step && q0 == qa && ncon + q0 >= 1 &&
                  (ncon + q0 <= 32 || (nwcon == 0 && ctx->world == 1 &&
                                       ncon + q0 + 1 <= PCU_MAX_COLS));
    wide_rhs = rhs_in_gram && ncon + q0 > 32;
  }
  const int nref = opt.iterative_refinement_steps;
  // fraction-to-boundary parameter of this iteration (IP.cpp:5069-5077), known before
  // the solves
  double tau_pre = opt.min_fraction_to_boundary;
  if (1.0 - barrier_param >= tau_pre) tau_pre = 1.0 - barrier_param;
  // The default iteration's solve: one refinement step done in the column space of
  // [A|Z], one pass (kktChain).  Its dense algebra runs on the device by default on one
  // GPU; across GPUs the host is faster (measured at 8 GPUs with the earlier two-pass
  // chain: 1.94 against 2.04 ms per iteration), so the device is taken there only on
  // request (PCU_CHAIN=1).  PCU_NO_FUSE21 / PCU_NO_FUSE2S select the elementwise
  // refinement of the two-pass route below.
  const bool colref = !inexact_newton_step && rhs_in_gram && !wide_rhs && nref == 1 &&
                      !mehrotra && !opt_no_fuse21 && !opt_no_fuse2s;
  const bool chain = colref && !opt_no_chain && ctx->chain_ok() &&
                     (ctx->world == 1 || opt_force_chain);
  if (opt.use_diag_hessian && (!colref || !hdiag || qn)) {
    // (the other routes would miss the Hessian term of their refinement residual; the
    // option has to be set before begin)
    if (ctx->rank == 0)
      fprintf(stderr, "ParOpt error: use_diag_hessian: this iteration is not on the route "
                      "of the column-space refinement, or the option was set after begin\n");
    return 1;
  }
  if (inexact_newton_step) {
    // nothing to set up
  } else if (colref) {
    if (kktChain(v, res, upd, use_qn, mu_for_res, tau_pre, VTp.data(), chain)) return 1;
  } else if (rhs_in_gram) {
    if (setUpKKTDiagRhs(v, use_qn, mu_for_res)) return 1;
    if (setUpKKTSystem(v, use_qn, nullptr, 1)) return 1;
  } else {
    if (setUpKKTDiagSystem(v, use_qn, 0)) return 1;
    if (setUpKKTSystem(v, use_qn, nullptr)) return 1;
  }
  if (diagonal_qn_step) use_qn = 0;
  auto kkt_with_refinement = [&](double mu_res, bool allow_refine) -> int {
    const int nr = allow_refine ? nref : 0;
    int emitted = 0;
    // after an inexact-Newton step the refinement residual takes the exact Hessian
    // (addKKTResStep with the outer flag, IP.cpp:5155-5156, 1461-1463)
    const bool hres = inexact_newton_step != 0;
    if (computeKKTStep(v, res, upd, use_qn, 0, VTp.data(), nr > 0 && !hres, mu_res, &emitted))
      return 1;
    for (int it = 0; it < nr; it++) {  // IP.cpp:4985-4991
      if (hres) {
        res_skip_hessian = 1;
        const int rc = computeKKTRes(v, mu_res, res, &upd, VTp.data(), VTp.data() + nA);
        res_skip_hessian = 0;
        if (rc || evalHvecProduct(upd.v[PCU_X], t1) ||
            pcu_vec_axpy(res.v[PCU_X], -1.0, t1))
          return 1;
        if (computeKKTStep(v, res, upd, use_qn, 1, VTp.data(), 0, mu_res, &emitted)) return 1;
        continue;
      }
      if (!emitted &&
          computeKKTRes(v, mu_res, res, &upd, VTp.data(), VTp.data() + nA))
        return 1;
      if (computeKKTStep(v, res, upd, use_qn, 1, VTp.data(), it + 1 < nr, mu_res,
                         &emitted))
        return 1;
    }
    return 0;
  };
  if (!colref && !inexact_newton_step) {
    // the fraction-to-boundary parameter is known before the solves (it depends on
    // the barrier only, IP.cpp:5069-5077), so the last pass of the last solve can
    // take the step statistics (not under the Mehrotra strategies, whose
    // predictor step is only a probe)
    double tau_s = -1.0;
    if (!mehrotra) {
      tau_s = opt.min_fraction_to_boundary;
      if (1.0 - barrier_param >= tau_s) tau_s = 1.0 - barrier_param;
    }
    // first step without refinement timing split: KKT solve = setup + first step
    int emitted = 0;
    if (computeKKTStep(v, res, upd, use_qn, 0, VTp.data(), nref > 0, mu_for_res,
                       &emitted, lazy_res ? 1 : 0, nref == 0 ? tau_s : -1.0))
      return 1;
    PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].k1, ctx->stream));
    for (int it = 0; it < nref; it++) {
      if (!emitted &&
          computeKKTRes(v, mu_for_res, res, &upd, VTp.data(), VTp.data() + nA))
        return 1;
      if (computeKKTStep(v, res, upd, use_qn, 1, VTp.data(), it + 1 < nref,
                         mu_for_res, &emitted, 0, it + 1 == nref ? tau_s : -1.0))
        return 1;
    }
  }
  (void)ref;
  double sums[StatsF::NS], mins[2];
  if (mehrotra && !inexact_newton_step) {  // IP.cpp:4999-5051
    if (stepStats(v, upd, 1.0, sums, mins)) return 1;
    const double max_x = mins[0], max_z = mins[1];
    double product = (sums[0] + max_x * sums[1] + max_z * sums[2] +
                      max_x * max_z * sums[3]) / opt.rel_bound_barrier +
                     (sums[4] + max_x * sums[5] + max_z * sums[6] +
                      max_x * max_z * sums[7]);
    double count = res_sums[1];
    for (int i = 0; i < ncon; i++) {
      product += (v.s[i] + max_x * upd.s[i]) * (v.zs[i] + max_z * upd.zs[i]) +
                 (v.t[i] + max_x * upd.t[i]) * (v.zt[i] + max_z * upd.zt[i]);
      count += 2.0;
    }
    const double comp_affine = count != 0.0 ? product / count : 0.0;
    const double s1 = comp_affine / comp;
    double sigma = s1 * s1 * s1;
    if (sigma < 0.01) sigma = 0.01;
    barrier_param = sigma * comp;
    if (barrier_param < 0.09999 * abs_res_tol) barrier_param = 0.09999 * abs_res_tol;
    if (computeKKTRes(v, barrier_param, res, nullptr, nullptr, nullptr)) return 1;
    computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
    // predictor-corrector: second-order terms of the affine step; the corrected
    // residual cannot be refined (IP.cpp:5029-5051)
    const bool mpc = ls.barrier_strategy == BS_MPC;
    if (mpc && addMehrotraCorrectorResidual(upd, res)) return 1;
    if (kkt_with_refinement(barrier_param, !mpc)) return 1;
  }

  // fraction to the boundary (IP.cpp:5069-5077)
  double tau = opt.min_fraction_to_boundary;
  if (1.0 - barrier_param >= tau) tau = 1.0 - barrier_param;

  double alpha_x = 1.0, alpha_z = 1.0;
  int ceq_step = 0;
  double m0 = 0.0, dm0 = 0.0;
  double pnorm2 = 0.0, px_maxabs_scaled = 0.0;

  // scaleKKTStep (IP.cpp:3196-3274) + evalMeritInitDeriv (IP.cpp:3652-3924) from
  // ONE statistics pass; the step itself stays unscaled on the device.
  auto scale_and_merit = [&](int inexact) -> int {
    StepScale sc;
    if (scaleAndMerit(v, upd, tau, comp, VTp.data(), -1.0, &sc, inexact)) return 1;
    alpha_x = sc.alpha_x;
    alpha_z = sc.alpha_z;
    ceq_step = sc.ceq;
    m0 = sc.m0;
    dm0 = sc.dm0;
    pnorm2 = sc.pnorm2;
    return 0;
  };
  if (scale_and_merit(inexact_newton_step)) return 1;

  double alpha = 1.0;
  int line_fail = LS_FAILURE;
  int update_type = 0;
  int line_search_skipped = 0;
  ls.no_merit_function_improvement = 0;

  // The first pass of computeStepAndUpdate (IP.cpp:4178-4216) from the step scaled by
  // ax, az; z_new: the new dense multipliers
  const bool form_pair = qn && uq;
  auto launch_update1 = [&](auto f1, double ax, double az, const double *z_new) -> int {
    f1.v = v.dv();
    f1.p = upd.dv();
    f1.lb = lb->d;
    f1.ub = ub->d;
    f1.g = g->d;
    f1.ncon = ncon;
    for (int j = 0; j < ncon; j++) {
      f1.Acol.p[j] = Ac[j]->d;
      f1.z.v[j] = z_new[j];
    }
    f1.yqn = form_pair ? y_qn->d : nullptr;
    if (form_pair && gaz_valid && apz_state == 3 && apz1 && apz2) {
      // -(g - A z+) = -(g - A z) + az A p_z: g - A z was left by the last update pass,
      // A p_z by the two pass-2 kernels of this iteration's solves -- three vectors
      // instead of g and the ncon constraint gradients
      f1.g = gaz->d;
      f1.ncon = 2;
      f1.Acol.p[0] = apz1->d;
      f1.Acol.p[1] = apz2->d;
      f1.z.v[0] = az;
      f1.z.v[1] = az;
    }
    f1.ax = ax;
    f1.az = az;
    f1.k = kconst();
    if (decltype(f1)::NS > 0) {
      RedBuf rb = ctx->redbuf(decltype(f1)::NS, decltype(f1)::NX, decltype(f1)::NM);
      if (launch_tile(ctx, f1, nvars, wd, rb)) return 1;
      ctx->defer();  // fetched together with Update2F's dots (or a callback's sums)
      return 0;
    }
    return launch_tile(ctx, f1, nvars, wd, NO_RED);
  };
  // The line search's first trial ran as TrialUpdateF and was accepted: the update pass
  // is done, its results wait in the trial buffers, and the next iteration's residual
  // statistics (Update1FT<1>'s, fetched with the merit sums) in trial_u1.
  int trial_updated = 0;
  double trial_u1[9];

  // computeStepAndUpdate (IP.cpp:4169-4267)
  auto step_and_update = [&](double a, int eval_obj_con) -> int {
    const double ax = a * alpha_x, az = a * alpha_z;
    for (int i = 0; i < ncon; i++) {  // dense parts (IP.cpp:4190-4194)
      const double dp = opt.design_precision;
      auto clip0 = [&](double x0, double st, double p) {
        double r = x0 + st * p;
        if (r <= dp) r = dp;
        return r;
      };
      v.s[i] = clip0(v.s[i], ax, upd.s[i]);
      v.t[i] = clip0(v.t[i], ax, upd.t[i]);
      v.z[i] = v.z[i] + az * upd.z[i];
      v.zs[i] = clip0(v.zs[i], az, upd.zs[i]);
      v.zt[i] = clip0(v.zt[i], az, upd.zt[i]);
    }
    // With a quasi-Newton pair to form, the infinity norm and the monotone strategy,
    // the two update passes also take the residual statistics of the NEXT iteration
    // at the new point (Update1FT<1> / Update2FT<1>): its stand-alone residual pass
    // and one synchronisation disappear.
    const bool take_stats = form_pair && lazy_res && norm_type_id() == 0 && !opt_no_updstats;
    if (trial_updated) {
      // the trial buffers become the variables (exchanged: the handles keep their
      // identity); the bound multipliers only where the pass wrote them
      if (pcu_vec_take(v.v[PCU_X], rx) ||
          (prob->use_lower && pcu_vec_take(v.v[PCU_ZL], rzl)) ||
          (prob->use_upper && pcu_vec_take(v.v[PCU_ZU], rzu)) ||
          pcu_vec_take(v.v[PCU_ZW], rzw) || pcu_vec_take(v.v[PCU_SW], rsw) ||
          pcu_vec_take(v.v[PCU_TW], rtw) || pcu_vec_take(v.v[PCU_ZSW], rzsw) ||
          pcu_vec_take(v.v[PCU_ZTW], rztw))
        return 1;
    } else if (take_stats ? launch_update1(Update1FT<1>(), ax, az, v.z.data())
                          : launch_update1(Update1FT<0>(), ax, az, v.z.data())) {
      return 1;
    }
    if (eval_obj_con) {
      if (evalObjCon(v.v[PCU_X])) {
        fprintf(stderr, "ParOpt: Function and constraint evaluation failed\n");
        return 1;
      }
    }
    // the new point is bit-identical to the one the objective callback saw last:
    // either x itself (eval_obj_con) or the accepted line-search trial point
    // (step_clip is the one definition of both)
    if (evalObjConGradient(v.v[PCU_X], 1)) {
      fprintf(stderr, "ParOpt: Gradient evaluation failed at final line search\n");
    }
    update_type = 0;
    if (qn) {
      if (uq) {
        double dots[3];
        auto launch_update2 = [&](auto f2) -> int {
          f2.zw = v.v[PCU_ZW]->d;
          f2.px = upd.v[PCU_X]->d;
          f2.g = g->d;
          f2.zl = prob->use_lower ? v.v[PCU_ZL]->d : nullptr;
          f2.zu = prob->use_upper ? v.v[PCU_ZU]->d : nullptr;
          f2.ncon = ncon;
          for (int j = 0; j < ncon; j++) {
            f2.Acol.p[j] = Ac[j]->d;
            f2.z.v[j] = v.z[j];
          }
          f2.yqn = y_qn->d;
          f2.sqn = s_qn->d;
          f2.ax = ax;
          // with three or more dense constraints: leave g - A z for the next solve
          if (ncon >= 3 && !opt_no_gaz) {
            if (!gaz) gaz = pcu_vec_create(ctx, nvars);
            if (!gaz) return 1;
            f2.gaz = gaz->d;
          }
          RedBuf rb = ctx->redbuf(3, decltype(f2)::NX, 0);
          if (launch_tile(ctx, f2, nvars, wd, rb)) return 1;
          gaz_valid = f2.gaz != nullptr;
          double out[4];
          if (ctx->fetch(out)) return 1;
          dots[0] = out[0];
          dots[1] = out[1];
          dots[2] = out[2];
          if (decltype(f2)::NX > 0) {
            // residual statistics of the next iteration, in ResF's layout
            double u1[9];
            if (trial_updated) memcpy(u1, trial_u1, sizeof(u1));
            else if (ctx->take_deferred(u1, 9)) return 1;
            memset(upd_sums, 0, sizeof(upd_sums));
            upd_sums[0] = u1[0];
            upd_sums[1] = u1[1];
            upd_sums[2] = u1[2];
            upd_max[0] = out[3];  // |rx|
            upd_max[1] = u1[3];   // |rzw|
            upd_max[2] = u1[4];   // |rsw|, |rtw|
            upd_max[3] = u1[5];   // bound products
            upd_max[4] = u1[6];   // sparse products
            upd_min[0] = u1[7];
            upd_min[1] = u1[8];
            upd_stats_valid = 1;
          }
          return 0;
        };
        // (more than 16 constraint gradients: 128-row tiles, so that the staged ring holds them)
        int rc2;
        if (ncon > 16)
          rc2 = take_stats ? launch_update2(Update2FT<1, 128>()) : launch_update2(Update2FT<0, 128>());
        else
          rc2 = take_stats ? launch_update2(Update2FT<1>()) : launch_update2(Update2FT<0>());
        if (rc2) return 1;
        // computeQuasiNewtonUpdateCorrection (IP.cpp:4258): the user may change
        // s and y, so the three dots are taken again afterwards
        const bool corrected = prob->hasQnUpdateCorrection();
        if (corrected) {
          if (prob->qnUpdateCorrection(v.v[PCU_X], v.z.data(), v.v[PCU_ZW], s_qn, y_qn)) return 1;
          if (pcu_vec_dot(y_qn, y_qn, &dots[0]) || pcu_vec_dot(y_qn, s_qn, &dots[1]) ||
              pcu_vec_dot(s_qn, s_qn, &dots[2]))
            return 1;
        }
        // s.S_i and s.Y_i: s = ax * p, so they are ax * (Z^T p) for L-BFGS
        std::vector<double> sZ;
        if (qn->type == 0 && !force_direct_dots && vtp_valid && !corrected) {
          sZ.resize(qn->size());
          for (int i = 0; i < qn->size(); i++) sZ[i] = ax * VTp[nA + i];
        }
        // s_qn / y_qn are rewritten from scratch by the next iteration: hand their
        // buffers to the quasi-Newton memory instead of copying them
        if (qn->update(s_qn, y_qn, dots[0], dots[1], dots[2],
                       sZ.empty() ? nullptr : sZ.data(), &update_type, 1))
          return 1;
      }
    }
    return 0;
  };

  // lineSearch (IP.cpp:3939-4156)
  auto line_search = [&](double alpha_min) -> int {
    int fail = LS_FAILURE;
    double merit = 0.0, best_merit = 0.0, best_alpha = -1.0;
    const int max_iters = opt.max_line_iters;
    std::vector<double> rs(ncon), rt(ncon);
    const double dp = opt.design_precision;
    // update: the trial is the update pass (TrialUpdateF), in case it is accepted
    auto eval_trial = [&](double a, bool merit_too, double *merit_out, bool update) -> int {
      if (update) {
        // spares of the multipliers the pass writes: 3W, and N per bound in use
        pcu_vec **wv[] = {&rzw, &rzsw, &rztw};
        for (auto pv : wv)
          if (!*pv && !(*pv = pcu_vec_create(ctx, nwcon))) return -1;
        if (prob->use_lower && !rzl && !(rzl = pcu_vec_create(ctx, nvars))) return -1;
        if (prob->use_upper && !rzu && !(rzu = pcu_vec_create(ctx, nvars))) return -1;
        TrialUpdateF fu;
        fu.r.x = rx->d;
        fu.r.zl = rzl ? rzl->d : nullptr;
        fu.r.zu = rzu ? rzu->d : nullptr;
        fu.r.zw = rzw->d;
        fu.r.sw = rsw->d;
        fu.r.tw = rtw->d;
        fu.r.zsw = rzsw->d;
        fu.r.ztw = rztw->d;
        const double az = a * alpha_z;
        std::vector<double> z_new(ncon);
        for (int i = 0; i < ncon; i++) z_new[i] = v.z[i] + az * upd.z[i];
        if (launch_update1(fu, a * alpha_x, az, z_new.data())) return -1;
      } else {
        TrialF ft;
        ft.v = v.dv();
        ft.p = upd.dv();
        ft.lb = lb->d;
        ft.ub = ub->d;
        ft.rx = rx->d;
        ft.rsw = rsw->d;
        ft.rtw = rtw->d;
        ft.ax = a * alpha_x;
        ft.k = kconst();
        RedBuf rb = ctx->redbuf(TrialF::NS, 0, 0);
        if (launch_tile(ctx, ft, nvars, wd, rb)) return -1;
        // the merit sums travel with the reductions the objective callback fetches
        // (one synchronisation for both)
        ctx->defer();
      }
      double ts[TrialF::NS];
      int fail_obj = evalObjCon(rx);
      if (update) {
        constexpr int TS = TrialUpdateF::TS, NS = TrialUpdateF::NS;
        double all[NS + TrialUpdateF::NX + TrialUpdateF::NM];
        if (ctx->take_deferred(all, NS + TrialUpdateF::NX + TrialUpdateF::NM)) return -1;
        for (int i = 0; i < TrialF::NS; i++) ts[i] = all[TS + i];
        // Update1FT<1>'s layout: its sums, then the maxima and minima
        for (int i = 0; i < TS; i++) trial_u1[i] = all[i];
        for (int i = 0; i < 9 - TS; i++) trial_u1[TS + i] = all[NS + i];
      } else if (ctx->take_deferred(ts, TrialF::NS)) {
        return -1;
      }
      if (fail_obj) return 1;
      if (!merit_too) return 0;
      for (int i = 0; i < ncon; i++) {
        double r = v.s[i] + a * alpha_x * upd.s[i];
        if (r <= dp) r = dp;
        rs[i] = r;
        r = v.t[i] + a * alpha_x * upd.t[i];
        if (r <= dp) r = dp;
        rt[i] = r;
      }
      // evalMeritFunc (IP.cpp:3524-3637)
      const double kap = opt.rel_bound_barrier;
      double pos = ts[0] * kap + ts[2], neg = ts[1] * kap + ts[3];
      double dense_infeas = 0.0;
      double m = fobj + ts[4];
      for (int i = 0; i < ncon; i++) {
        const double l1 = log(rs[i]), l2 = log(rt[i]);
        if (rs[i] > 1.0) pos += l1; else neg += l1;
        if (rt[i] > 1.0) pos += l2; else neg += l2;
        const double cval = c[i] - rs[i] + rt[i];
        dense_infeas += cval * cval;
      }
      const double infeas = sqrt(dense_infeas + ts[5]);
      m += -barrier_param * (pos + neg) + rho_penalty_search * infeas;
      for (int i = 0; i < ncon; i++) m += gamma_s[i] * rs[i] + gamma_t[i] * rt[i];
      *merit_out = m;
      return 0;
    };
    // the first trial is also the update pass unless the last line search rejected
    // its first trial
    const bool update_first = !opt_no_trialupd && !ls.first_trial_rejected;
    int j = 0;
    for (; j < max_iters; j++) {
      int rc = eval_trial(alpha, true, &merit, j == 0 && update_first);
      if (j == 0) ls.first_trial_rejected = 1;  // until the test below accepts it
      if (rc < 0) return -1;
      if (rc > 0) {
        fprintf(stderr,
                "ParOpt: Evaluation failed during line search, trying new point\n");
        alpha *= 0.1;
        continue;
      }
      if (best_alpha < 0.0 || merit < best_merit) {
        best_alpha = alpha;
        best_merit = merit;
      }
      if (merit - opt.armijo_constant * alpha * dm0 < m0 + fp) {
        if (fail & LS_MIN_STEP) fail = LS_SUCCESS | LS_MIN_STEP;
        else fail = LS_SUCCESS;
        if (merit <= m0 + fp && merit + fp >= m0) fail |= LS_NO_IMPROVEMENT;
        if (j == 0) {
          ls.first_trial_rejected = 0;
          trial_updated = update_first;
        }
        break;
      } else if (fail & LS_MIN_STEP) {
        break;
      }
      if (j < max_iters - 1) {
        if (opt.use_backtracking_alpha) {
          alpha = 0.5 * alpha;
          if (alpha <= alpha_min) {
            alpha = alpha_min;
            fail |= LS_MIN_STEP;
          }
        } else {
          const double alpha_new =
              -0.5 * dm0 * (alpha * alpha) / (merit - m0 - dm0 * alpha);
          if (alpha_new <= alpha_min) {
            alpha = alpha_min;
            fail |= LS_MIN_STEP;
          } else if (alpha_new < 0.01 * alpha) {
            alpha = 0.01 * alpha;
          } else {
            alpha = alpha_new;
          }
        }
      }
    }
    if (j == max_iters) fail |= LS_MAX_ITERS;
    if (!(fail & LS_SUCCESS)) {
      if (best_merit <= m0 + fp) {
        fail |= LS_SUCCESS;
        fail &= ~LS_FAILURE;
      } else if (merit <= m0 + fp && merit + fp >= m0) {
        fail |= LS_NO_IMPROVEMENT;
      }
      if (alpha != best_alpha) {
        alpha = best_alpha;
        double dummy;
        int rc = eval_trial(alpha, false, &dummy, false);
        if (rc != 0) {
          fprintf(stderr, "ParOpt: Evaluation failed during line search\n");
          fail = LS_FAILURE;
        }
      }
    }
    return fail;
  };

  if (opt.use_line_search) {
    ls.dm0_prev = dm0;
    if (dm0 >= 0.0 && dm0 <= fp) {
      line_search_skipped = 1;
      if (step_and_update(alpha, 1)) return 1;
      if ((ls.fobj_prev + fp <= fobj) && (fobj + fp <= ls.fobj_prev))
        line_fail = LS_NO_IMPROVEMENT;
    } else {
      if (dm0 >= 0.0) {  // IP.cpp:5130-5173
        if (hess_obj) {
          qn_hessian_reset = 1;
          if (qn) qn->reset();
        }
        if (computeKKTRes(v, barrier_param, res, nullptr, nullptr, nullptr)) return 1;
        computeResNorm(res, &max_prime, &max_dual, &max_infeas, &res_norm);
        diagonal_qn_step = 1;
        use_qn = 1;
        if (opt.use_diag_hessian) {
          // the same solve on the route this option runs on (its refinement residual
          // carries h; the two-pass route's would not)
          if (kktChain(v, res, upd, use_qn, barrier_param, tau, VTp.data(), chain)) return 1;
        } else {
          if (setUpKKTDiagSystem(v, use_qn, 0)) return 1;
          if (setUpKKTSystem(v, use_qn, nullptr)) return 1;
          if (kkt_with_refinement(barrier_param, true)) return 1;
        }
        if (scale_and_merit(0)) return 1;
        ls.dm0_prev = dm0;
      }
      if (dm0 >= 0.0) {
        line_fail = LS_FAILURE;
      } else {
        // px_norm is the max-abs of the alpha_x-scaled step (IP.cpp:5183)
        px_maxabs_scaled = alpha_x * stats_pmax;
        double alpha_min = 1.0;
        if (px_maxabs_scaled != 0.0) alpha_min = fp / px_maxabs_scaled;
        if (alpha_min > 0.5) alpha_min = 0.5;
        line_fail = line_search(alpha_min);
        if (line_fail < 0) return 1;
        if (px_maxabs_scaled < opt.design_precision) line_fail |= LS_SHORT_STEP;
        if (!(line_fail & LS_FAILURE)) {
          if (step_and_update(alpha, 0)) return 1;
        }
      }
    }
  } else {
    ls.dm0_prev = dm0;
    line_fail = LS_SUCCESS;
    if (step_and_update(alpha, 1)) return 1;
    // merit at the new point (IP.cpp:5236-5243): trial kernel with zero step
    TrialF ft;
    ft.v = v.dv();
    ft.p = upd.dv();
    ft.lb = lb->d;
    ft.ub = ub->d;
    ft.rx = rx->d;
    ft.rsw = rsw->d;
    ft.rtw = rtw->d;
    ft.ax = 0.0;
    ft.k = kconst();
    RedBuf rb = ctx->redbuf(TrialF::NS, 0, 0);
    if (launch_tile(ctx, ft, nvars, wd, rb)) return 1;
    double ts[TrialF::NS];
    if (ctx->fetch(ts)) return 1;
    const double kap = opt.rel_bound_barrier;
    double pos = ts[0] * kap + ts[2], neg = ts[1] * kap + ts[3];
    double dense_infeas = 0.0;
    double m1 = fobj + ts[4];
    for (int i = 0; i < ncon; i++) {
      const double l1 = log(v.s[i]), l2 = log(v.t[i]);
      if (v.s[i] > 1.0) pos += l1; else neg += l1;
      if (v.t[i] > 1.0) pos += l2; else neg += l2;
      const double cval = c[i] - v.s[i] + v.t[i];
      dense_infeas += cval * cval;
      m1 += gamma_s[i] * v.s[i] + gamma_t[i] * v.t[i];
    }
    m1 += -barrier_param * (pos + neg) +
          rho_penalty_search * sqrt(dense_infeas + ts[5]);
    if (m1 <= m0 + fp && m1 + fp >= m0) line_fail |= LS_NO_IMPROVEMENT;
    else if (fabs(dm0) <= fp) line_fail = LS_NO_IMPROVEMENT;
  }

  ls.no_merit_function_improvement =
      ((line_fail & LS_NO_IMPROVEMENT) || (line_fail & LS_MIN_STEP) ||
       (line_fail & LS_SHORT_STEP) || (line_fail & LS_FAILURE)) ? 1 : 0;
  ls.line_search_failed = (line_fail & LS_FAILURE);
  ls.alpha_prev = alpha;
  ls.alpha_xprev = alpha_x;
  ls.alpha_zprev = alpha_z;
  ls.last_pnorm2 = pnorm2;
  if (hess_obj && uq && (line_fail & LS_FAILURE)) {
    qn_hessian_reset = 1;
    if (qn) qn->reset();
  }
  std::string info;
  if (gmres_iters != 0) info += "iNK" + std::to_string(gmres_iters) + " ";
  if (update_type == 1) info += "dampH ";
  else if (update_type == 2) info += "skipH ";
  if (qn_hessian_reset) info += "resetH ";
  if (line_fail & LS_FAILURE) info += "LFail ";
  if (line_fail & LS_MIN_STEP) info += "LMnStp ";
  if (line_fail & LS_MAX_ITERS) info += "LMxItr ";
  if (line_fail & LS_NO_IMPROVEMENT) info += "LNoImprv ";
  if (seq_linear_step) info += "SLP ";
  if (diagonal_qn_step) info += "DQN ";
  if (line_search_skipped) info += "LSkip ";
  if (ceq_step) info += "cmpEq ";
  while (!info.empty() && info.back() == ' ') info.pop_back();
  ls.info = info;
  if (monotone_barrier_converged) ls.barrier_strategy = ls.input_barrier_strategy;

  PCU_CUDA_OK(cudaEventRecord(evs[ev_cur].it1, ctx->stream));
  evs[ev_cur].pending = true;
  ls.k++;
  niter++;
  return 0;
}
