// pcu_kernels.cuh -- the fused interior-point kernels (functors for tile_kernel).
//
// Each functor restates one or more private methods of the reference's
// ParOptInteriorPoint (IP.cpp = /root/reference/src/ParOptInteriorPoint.cpp) as a
// single pass over the local design variables (N) and weighting constraints
// (W).  Algorithmic traffic per launch is stated with every functor
// ("words" = fp64 words; c = dense constraints, q = quasi-Newton width).
//
// Functor protocol (see tile_kernel in pcu_common.cuh):
//   A<W>(i, coef, elem, part)   loads W consecutive elements, returns the terms
//                               of the per-constraint block sums; idempotent
//   B(ci, sum, con, acc)        run by ONE thread per weighting constraint; the
//                               harness broadcasts con.d[] to the constraint's
//                               elements
//   C<W>(i, coef, elem, con, acc)  finishes the elements and stores
#pragma once

#include "pcu_common.cuh"
#include "pcu_dense.cuh"

// occupancy hints (blocks of 128 threads per SM) of the register-heavy kernels
#ifndef PCU_MINB_RES
#define PCU_MINB_RES 5
#endif
#ifndef PCU_MINB_STATS
#define PCU_MINB_STATS 5
#endif
#ifndef PCU_MINB_PASS1
#define PCU_MINB_PASS1 5
#endif
#ifndef PCU_MINB_PASS21
#define PCU_MINB_PASS21 6
#endif
#ifndef PCU_MINB_PASS2S
#define PCU_MINB_PASS2S 7
#endif
#ifndef PCU_SMEMACC21
#define PCU_SMEMACC21 1
#endif

struct DVars {  // device view of ParOptVars (IP.h:373-389)
  double *x, *zl, *zu;               // N
  double *zw, *sw, *tw, *zsw, *ztw;  // W
};

struct IPConst {
  double mbv;     // max_bound_value
  double kappa;   // rel_bound_barrier
  double gamma;   // penalty_gamma: gamma_tw = gamma, gamma_sw = gamma for sparse
                  // equalities and 0 for sparse inequalities (IP.cpp:357-374)
  double dp;      // design_precision
  double wconst;  // constant term of cw(x)
  // per-constraint constant terms (null: wconst for every row).  The trust-region
  // subproblem's sparse constraints are cw(x_k) + Aw p (ParOptTrustRegion.cpp:318-321):
  // the same rows, a different constant each.
  const double *wc;
  int use_lower, use_upper;
  int nwineq;     // local number of sparse inequalities
};

__device__ __forceinline__ double wconst_at(const IPConst &k, long long ci) {
  return k.wc ? k.wc[ci] : k.wconst;
}
__device__ __forceinline__ double gamma_sw(const IPConst &k, long long ci) {
  return ci < k.nwineq ? 0.0 : k.gamma;
}

// Coefficient j of a column table: from kernel-parameter space (host-computed), or --
// device chain of the KKT solve, pcu_dense.cu -- from a constant bank that a
// stream-ordered device-to-device copy fills from the dense kernel's output right
// before this launch (cudaMemcpyToSymbolAsync): the same constant-cache operand either
// way, no load in the column loops.  Layout: alpha of Pass2SVF (pcu_dense_solve).
// (One bank per device and process: the chain is only taken while a single context
// uses the device, pcu_ctx::chain_ok.)
static __constant__ double pcu_chain_coef[PCU_DENSE_MAXM];
__device__ __forceinline__ double pcu_coef(int cbank, const CoefTable &tab, int j) {
  return cbank >= 0 ? pcu_chain_coef[cbank + j] : tab.v[j];
}

struct Con0 {  // no per-constraint data
  static constexpr int ND = 0;
  double d[1];
  __device__ __forceinline__ void zero() {}
};
struct Con2 {  // two broadcast values
  static constexpr int ND = 2;
  double d[2];
  __device__ __forceinline__ void zero() { d[0] = d[1] = 0.0; }
};
struct Con1 {  // one broadcast value
  static constexpr int ND = 1;
  double d[1];
  __device__ __forceinline__ void zero() { d[0] = 0.0; }
};

// ============================================================== ResF
// computeKKTRes (IP.cpp:1337-1446) + computeResNorm (IP.cpp:1588-1723) +
// computeComp (IP.cpp:2742-2820) and, when has_step, addKKTResStep
// (IP.cpp:1451-1583) with the quasi-Newton product expanded through the compact
// form  B p = (b0 + sigma) p - sum_k kap_k Z_k.
// Traffic: reads (6 + c)N [+ (3 + q)N with step], writes 3N; W: 5r [+5r] + 5w.
// sums: 0 bound comp product, 1 comp count (bounds present + 2 per sparse
//       constraint), 2 sparse comp product,
//       3 norm-sum rx, 4 norm-sum rzw, 5..8 l1 of rsw,rtw,rzsw,rztw,
//       9,10 norm-sum rzl, rzu;   maxima: 0 |rx|, 1 |rzw|, 2 dual parts
// HS / NT fix has_step / norm_type at compile time (-1: run-time value): the
// per-iteration launch (no step terms, infinity norm) sheds a third of its
// instructions, and this pass is issue-bound, not bandwidth-bound.
template <int HS, int NT>
struct ResFT : NoStreams {
  __host__ __device__ __forceinline__ int hs() const { return HS < 0 ? has_step : HS; }
  __host__ __device__ __forceinline__ int nt() const { return NT < 0 ? norm_type : NT; }
  static constexpr int SRC = 1;
  static constexpr int MINB = PCU_MINB_RES;
  enum { S_X, S_LB, S_UB, S_G, S_ZL, S_ZU, S_PX, S_PZL, S_PZU, S_A0 };  // then A, then Z columns
  static constexpr int NFIX = S_A0;  // fixed slots; the columns follow
  static constexpr int TROWS = 512;
  enum { W_ZW, W_SW, W_TW, W_ZSW, W_ZTW, W_PZW, W_PSW, W_PTW, W_PZSW, W_PZTW, NWSLOTS };
  // maxima: 0 |rx|, 1 |rzw|, 2 mu-independent dual parts (|rsw|, |rtw|) and, for
  // l1/l2 bookkeeping, every dual part; 3 max zl(x-lb) | zu(ub-x); 4 max sw zsw |
  // tw ztw.  minima: 0 / 1 the same two products.  With them the infinity-norm
  // of the mu-dependent parts |kappa mu - a_i| is exact for ANY mu, so a barrier
  // update needs no second pass (IP.cpp:4726-4729).
  static constexpr int NS = 11, NX = 5, NM = 2, NB = 2;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // zw (+ pzw)
  struct Elem {
    double rx, rzl, rzu, cprod, ccount, amax, amin;
  };
  DVars v, r, p;
  const double *lb, *ub, *g;
  ColTable Acol;
  CoefTable z;  // dense multipliers z_j (+ pz_j when has_step, added on host)
  int ncon;
  ColTable Z;
  CoefTable kap;
  int nq;
  double b0sig;
  double mu;
  int has_step;
  int norm_type;  // 0 infinity, 1 l1, 2 l2
  int store;      // write the residual vectors (0: statistics only)
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(lb); p_(ub); p_(g);
    if (k.use_lower) p_(v.zl);
    if (k.use_upper) p_(v.zu);
    for (int j = 0; j < ncon; j++) p_(Acol.p[j]);
    if (hs()) {
      p_(p.x);
      if (k.use_lower) p_(p.zl);
      if (k.use_upper) p_(p.zu);
      for (int j = 0; j < nq; j++) p_(Z.p[j]);
    }
  }

  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_X, v.x); p_.n(S_LB, lb); p_.n(S_UB, ub); p_.n(S_G, g);
    if (k.use_lower) p_.n(S_ZL, v.zl);
    if (k.use_upper) p_.n(S_ZU, v.zu);
    for (int j = 0; j < ncon; j++) p_.n(S_A0 + j, Acol.p[j]);
    p_.w(W_ZW, v.zw); p_.w(W_SW, v.sw); p_.w(W_TW, v.tw); p_.w(W_ZSW, v.zsw);
    p_.w(W_ZTW, v.ztw);
    if (hs()) {
      p_.n(S_PX, p.x);
      if (k.use_lower) p_.n(S_PZL, p.zl);
      if (k.use_upper) p_.n(S_PZU, p.zu);
      for (int j = 0; j < nq; j++) p_.n(S_A0 + ncon + j, Z.p[j]);
      p_.w(W_PZW, p.zw); p_.w(W_PSW, p.sw); p_.w(W_PTW, p.tw); p_.w(W_PZSW, p.zsw);
      p_.w(W_PZTW, p.ztw);
    }
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void A(const S &src, long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][2], AT *acc) const {
    double x[W], l[W], u[W], zl[W], zu[W], gv[W], rx[W];
    src.template ld<W>(S_X, v.x, i, x);
    src.template ld<W>(S_LB, lb, i, l);
    src.template ld<W>(S_UB, ub, i, u);
    src.template ld<W>(S_G, g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = 0.0;
    if (k.use_lower) src.template ld<W>(S_ZL, v.zl, i, zl);
    if (k.use_upper) src.template ld<W>(S_ZU, v.zu, i, zu);
#pragma unroll
    for (int q = 0; q < W; q++) rx[q] = (zl[q] - zu[q]) - gv[q];
    for (int j = 0; j < ncon; j++) {
      double a[W];
      src.template ldc<W>(j, Acol.p[j], i, a);
#pragma unroll
      for (int q = 0; q < W; q++) rx[q] = fma(z.v[j], a[q], rx[q]);
    }
    double px[W], pzl[W], pzu[W];
#pragma unroll
    for (int q = 0; q < W; q++) px[q] = pzl[q] = pzu[q] = 0.0;
    if (hs()) {
      src.template ld<W>(S_PX, p.x, i, px);
      if (k.use_lower) src.template ld<W>(S_PZL, p.zl, i, pzl);
      if (k.use_upper) src.template ld<W>(S_PZU, p.zu, i, pzu);
#pragma unroll
      for (int q = 0; q < W; q++)
        rx[q] = fma(-b0sig, px[q], rx[q]) + (pzl[q] - pzu[q]);
      for (int j = 0; j < nq; j++) {
        double zc[W];
        src.template ldc<W>(ncon + j, Z.p[j], i, zc);
#pragma unroll
        for (int q = 0; q < W; q++) rx[q] = fma(kap.v[j], zc[q], rx[q]);
      }
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      const bool ml = k.use_lower && (l[q] > -k.mbv);
      const bool mu_ = k.use_upper && (u[q] < k.mbv);
      const double dl = x[q] - l[q], du = u[q] - x[q];
      double rzl = 0.0, rzu = 0.0, cp = 0.0, cc = 0.0;
      double amax = 0.0, amin = 1.0e300;
      if (ml) {
        const double a = dl * zl[q];
        rzl = -(a - k.kappa * mu);
        if (hs()) rzl -= (dl * pzl[q] + px[q] * zl[q]);
        cp += a;
        cc += 1.0;
        amax = fmax(amax, a);
        amin = fmin(amin, a);
      }
      if (mu_) {
        const double a = du * zu[q];
        rzu = -(a - k.kappa * mu);
        if (hs()) rzu -= (du * pzu[q] - px[q] * zu[q]);
        cp += a;
        cc += 1.0;
        amax = fmax(amax, a);
        amin = fmin(amin, a);
      }
      e[q].amax = amax;
      e[q].amin = amin;
      e[q].rx = rx[q];
      e[q].rzl = rzl;
      e[q].rzu = rzu;
      e[q].cprod = cp;
      e[q].ccount = cc;
      part[q][0] = coef[q] * x[q];
      part[q][1] = coef[q] * px[q];
    }
  }

  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&sum)[2],
                                    Con &con, AT &acc) const {
    const double zw = src.ldw(W_ZW, v.zw, ci), sw = src.ldw(W_SW, v.sw, ci), tw = src.ldw(W_TW, v.tw, ci);
    const double zsw = src.ldw(W_ZSW, v.zsw, ci), ztw = src.ldw(W_ZTW, v.ztw, ci);
    const double gsw = gamma_sw(k, ci), gtw = k.gamma;
    double rzw = -(((wconst_at(k, ci) + sum[0]) - sw) + tw);
    double rsw = (zsw - gsw) - zw;
    double rtw = (ztw - gtw) + zw;
    const double asw = sw * zsw, atw = tw * ztw;
    double rzsw = mu - asw;
    double rztw = mu - atw;
    acc.x[4] = fmax(acc.x[4], fmax(asw, atw));
    acc.m[1] = fmin(acc.m[1], fmin(asw, atw));
    con.d[0] = zw;
    if (hs()) {
      const double pzw = src.ldw(W_PZW, p.zw, ci), psw = src.ldw(W_PSW, p.sw, ci), ptw = src.ldw(W_PTW, p.tw, ci);
      const double pzsw = src.ldw(W_PZSW, p.zsw, ci), pztw = src.ldw(W_PZTW, p.ztw, ci);
      rzw += (psw - sum[1]) - ptw;
      rsw += pzsw - pzw;
      rtw += pztw + pzw;
      rzsw -= (psw * zsw + sw * pzsw);
      rztw -= (ptw * ztw + tw * pztw);
      con.d[0] += pzw;
    }
    if (store) {
      r.zw[ci] = rzw;
      r.sw[ci] = rsw;
      r.tw[ci] = rtw;
      r.zsw[ci] = rzsw;
      r.ztw[ci] = rztw;
    }
    acc.s[2] += asw + atw;
    acc.s[1] += 2.0;
    acc.x[1] = fmax(acc.x[1], fabs(rzw));
    acc.x[2] = fmax(acc.x[2], fmax(fabs(rsw), fabs(rtw)));
    if (hs())  // no closed form in mu once the step terms are in
      acc.x[2] = fmax(acc.x[2], fmax(fabs(rzsw), fabs(rztw)));
    if (nt() == 1) {
      acc.s[4] += fabs(rzw);
    } else if (nt() == 2) {
      acc.s[4] = fma(rzw, rzw, acc.s[4]);
    }
    if (nt() != 0) {
      acc.s[5] += fabs(rsw);
      acc.s[6] += fabs(rtw);
      acc.s[7] += fabs(rzsw);
      acc.s[8] += fabs(rztw);
    }
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void C(const S &, long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AT &acc) const {
    double rx[W], rzl[W], rzu[W];
#pragma unroll
    for (int q = 0; q < W; q++) {
      rx[q] = fma(coef[q], con.d[0], e[q].rx);  // + Aw^T (zw [+ pzw])
      rzl[q] = e[q].rzl;
      rzu[q] = e[q].rzu;
      acc.s[0] += e[q].cprod;
      acc.s[1] += e[q].ccount;
      acc.x[0] = fmax(acc.x[0], fabs(rx[q]));
      acc.x[3] = fmax(acc.x[3], e[q].amax);
      acc.m[0] = fmin(acc.m[0], e[q].amin);
      if (hs()) acc.x[2] = fmax(acc.x[2], fmax(fabs(rzl[q]), fabs(rzu[q])));
      if (nt() == 1) {
        acc.s[3] += fabs(rx[q]);
        acc.s[9] += fabs(rzl[q]);
        acc.s[10] += fabs(rzu[q]);
      } else if (nt() == 2) {
        acc.s[3] = fma(rx[q], rx[q], acc.s[3]);
        acc.s[9] = fma(rzl[q], rzl[q], acc.s[9]);
        acc.s[10] = fma(rzu[q], rzu[q], acc.s[10]);
      }
    }
    if (store) {
      stv<W>(r.x, i, rx);
      if (k.use_lower) stv<W>(r.zl, i, rzl);
      if (k.use_upper) stv<W>(r.zu, i, rzu);
    }
  }
};
typedef ResFT<-1, -1> ResF;

// ============================================================== DiagF
// setUpKKTDiagSystem, diagonal part (IP.cpp:1864-1927) + ParOptQuasiDefBlockMat
// ::factor with nwblock = 1 (SM.cpp:41-115): Dinv and Cw = 1/(Cdiag + Aw Dinv
// Aw^T).  identity != 0 gives the matrices of initLeastSquaresMultipliers
// (IP.cpp:5418-5431): Dinv = 1, Cdiag = small.
// Traffic: reads 5N + 4W, writes N + W.
//
// HD = 1 (use_diag_hessian): the Hessian block is diag(h) + sigma, the problem's
// diagonal (evalHessianDiag) in place of b0 + Z M Z^T; b0sig is then sigma alone.
// One more N-stream: reads 6N + 4W.  The h pointer exists in the HD = 1 types only, so
// the HD = 0 kernels keep their parameter blocks and their code.
template <int HD> struct HessDiagPtr { const double *h; };
template <> struct HessDiagPtr<0> {};
template <int HD>
struct DiagFT : NoStreams, HessDiagPtr<HD> {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  DVars v;
  const double *lb, *ub;
  double *Dinv, *Cw;
  double b0sig;
  int identity;
  double small_;
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    if (!identity) {
      p_(v.x); p_(lb); p_(ub);
      if (k.use_lower) p_(v.zl);
      if (k.use_upper) p_(v.zu);
      if constexpr (HD) p_(this->h);
    }
  }

  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W],
                                    Elem (&)[W], double (&part)[W][1], AccT *acc) const {
    double d[W];
    if (identity) {
#pragma unroll
      for (int q = 0; q < W; q++) d[q] = 1.0;
    } else {
      double x[W], l[W], u[W], zl[W], zu[W], hv[W];
      ldv<W>(v.x, i, x);
      ldv<W>(lb, i, l);
      ldv<W>(ub, i, u);
#pragma unroll
      for (int q = 0; q < W; q++) zl[q] = zu[q] = 0.0;
      if (k.use_lower) ldv<W>(v.zl, i, zl);
      if (k.use_upper) ldv<W>(v.zu, i, zu);
      if constexpr (HD) ldv<W>(this->h, i, hv);
#pragma unroll
      for (int q = 0; q < W; q++) {
        double t = b0sig;
        if constexpr (HD) t = hv[q] + b0sig;
        if (k.use_lower && l[q] > -k.mbv) t += zl[q] / (x[q] - l[q]);
        if (k.use_upper && u[q] < k.mbv) t += zu[q] / (u[q] - x[q]);
        d[q] = 1.0 / t;
      }
    }
    stv<W>(Dinv, i, d);
#pragma unroll
    for (int q = 0; q < W; q++) part[q][0] = coef[q] * coef[q] * d[q];
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1], Con &,
                                    AccT &) const {
    double cdiag = small_;
    if (!identity) cdiag = v.sw[ci] / v.zsw[ci] + v.tw[ci] / v.ztw[ci];
    Cw[ci] = 1.0 / (cdiag + sum[0]);
  }
  template <int W>
  __device__ __forceinline__ void C(long long, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {}
};
// distinct types, so that kernel names and profiles tell the two apart
struct DiagF : DiagFT<0> {};
struct DiagHF : DiagFT<1> {};

// ============================================================== BlockFactorF / BlockApplyF
// ParOptQuasiDefBlockMat with nwblock = 1 as a stand-alone object (SM.cpp:41-224):
// factor: Cw = 1 / (Cdiag + Aw Dinv Aw^T) (a zero pivot is reported, :91-98);
// apply:  yw = Cw (bw - Aw Dinv bx) [bw = 0 in the 3-argument form],
//         yx = Dinv (bx + Aw^T yw)   -- the reference's sign convention (:117-190).
// Traffic: factor N + 2W; apply 3N + 3W (4-argument form), one pass each.
struct BlockFactorF : NoStreams {
  static constexpr int NS = 0, NX = 1, NM = 0, NB = 1;  // max: failing row + 1
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *Dinv, *Cdiag;
  double *Cw;
  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W], Elem (&)[W],
                                    double (&part)[W][1], AccT *) const {
    double d[W];
    ldv<W>(Dinv, i, d);
#pragma unroll
    for (int q = 0; q < W; q++) part[q][0] = coef[q] * coef[q] * d[q];
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1], Con &,
                                    AccT &acc) const {
    const double e = Cdiag[ci] + sum[0];
    if (e == 0.0) {
      acc.x[0] = fmax(acc.x[0], (double)(ci + 1));
      Cw[ci] = 0.0;
    } else {
      Cw[ci] = 1.0 / e;
    }
  }
  template <int W>
  __device__ __forceinline__ void C(long long, const double (&)[W], const Elem (&)[W],
                                    const Con &, AccT &) const {}
};
struct BlockApplyF : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // yw
  struct Elem {
    double bx, dinv;
  };
  const double *bx, *bw, *Dinv, *Cw;  // bw may be null (3-argument apply)
  double *yx, *yw;
  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W], Elem (&e)[W],
                                    double (&part)[W][1], AccT *) const {
    double b[W], d[W];
    ldv<W>(bx, i, b);
    ldv<W>(Dinv, i, d);
#pragma unroll
    for (int q = 0; q < W; q++) {
      e[q].bx = b[q];
      e[q].dinv = d[q];
      part[q][0] = coef[q] * (d[q] * b[q]);
    }
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1], Con &con,
                                    AccT &) const {
    const double r = (bw ? bw[ci] : 0.0) - sum[0];
    const double v = r * Cw[ci];
    yw[ci] = v;
    con.d[0] = v;
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con, AccT &) const {
    double o[W];
#pragma unroll
    for (int q = 0; q < W; q++) o[q] = fma(coef[q], con.d[0], e[q].bx) * e[q].dinv;
    stv<W>(yx, i, o);
  }
};

// ============================================================== DiagRhsF
// DiagF fused with the right-hand side of the iteration's first diagonal solve:
// d1, d2 of solveKKTDiagSystem (IP.cpp:2091-2139) applied to the KKT residual
// itself (computeKKTRes, IP.cpp:1337-1446, at barrier mu), recomputed from the
// variables exactly as Pass1VF does.  The solve's block part and the products
// [A|Z]^T t1 then ride along in the Gram pass as one more column (pcu_gram.cu),
// so the first solve of an iteration has no pass 1 of its own.
// Traffic: reads (6 + c)N + 5W, writes 2N + 2W.
// HD = 1 (DiagRhsHF, use_diag_hessian): c = h_i + sigma, as DiagFT<1>; reads (7 + c)N.
template <int HD>
struct DiagRhsFT : NoStreams, HessDiagPtr<HD> {
  static constexpr int SRC = 1;
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 2, HASP = 1;
  enum { S_X, S_LB, S_UB, S_G, S_ZL, S_ZU, S_H };
  static constexpr int S_A0 = S_H + HD;
  static constexpr int NFIX = S_A0;  // fixed slots; the columns follow
  static constexpr int TROWS = 512;
  enum { W_ZW, W_SW, W_TW, W_ZSW, W_ZTW, NWSLOTS };
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // zw
  struct Elem {};
  DVars v;
  const double *lb, *ub, *g;
  double *Dinv, *Cw, *d1, *d2;
  ColTable Acol;
  CoefTable z;
  int ncon;
  double b0sig, mu;
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(lb); p_(ub); p_(g);
    if (k.use_lower) p_(v.zl);
    if (k.use_upper) p_(v.zu);
    if constexpr (HD) p_(this->h);
    for (int j = 0; j < ncon; j++) p_(Acol.p[j]);
  }
  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_X, v.x); p_.n(S_LB, lb); p_.n(S_UB, ub); p_.n(S_G, g);
    if (k.use_lower) p_.n(S_ZL, v.zl);
    if (k.use_upper) p_.n(S_ZU, v.zu);
    if constexpr (HD) p_.n(S_H, this->h);
    for (int j = 0; j < ncon; j++) p_.n(S_A0 + j, Acol.p[j]);
    p_.w(W_ZW, v.zw); p_.w(W_SW, v.sw); p_.w(W_TW, v.tw); p_.w(W_ZSW, v.zsw);
    p_.w(W_ZTW, v.ztw);
  }
  template <class S>
  __device__ __forceinline__ void P(const S &src, long long ci, Con &con) const {
    con.d[0] = src.ldw(W_ZW, v.zw, ci);
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void AP(const S &src, long long i, const double (&coef)[W],
                                     Elem (&)[W], double (&part)[W][2], AT *,
                                     const Con &con) const {
    double x[W], l[W], u[W], gv[W], zl[W], zu[W], di[W], d[W];
    src.template ld<W>(S_X, v.x, i, x);
    src.template ld<W>(S_LB, lb, i, l);
    src.template ld<W>(S_UB, ub, i, u);
    src.template ld<W>(S_G, g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = 0.0;
    if (k.use_lower) src.template ld<W>(S_ZL, v.zl, i, zl);
    if (k.use_upper) src.template ld<W>(S_ZU, v.zu, i, zu);
    double hv[W];
    if constexpr (HD) src.template ld<W>(S_H, this->h, i, hv);
#pragma unroll
    for (int q = 0; q < W; q++) d[q] = (zl[q] - zu[q]) - gv[q];
    for (int j = 0; j < ncon; j++) {
      double a[W];
      src.template ldc<W>(j, Acol.p[j], i, a);
#pragma unroll
      for (int q = 0; q < W; q++) d[q] = fma(z.v[j], a[q], d[q]);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      const double dl = x[q] - l[q], du = u[q] - x[q];
      double c = b0sig;                           // IP.cpp:1864-1910
      if constexpr (HD) c = hv[q] + b0sig;
      double t = fma(coef[q], con.d[0], d[q]);    // rx
      if (k.use_lower && l[q] > -k.mbv) {
        const double rl = pcu_rcp(dl);
        c = fma(zl[q], rl, c);
        t += -(dl * zl[q] - k.kappa * mu) * rl;
      }
      if (k.use_upper && u[q] < k.mbv) {
        const double ru = pcu_rcp(du);
        c = fma(zu[q], ru, c);
        t -= -(du * zu[q] - k.kappa * mu) * ru;
      }
      di[q] = pcu_rcp(c);
      d[q] = t;
      part[q][0] = coef[q] * coef[q] * di[q];
      part[q][1] = coef[q] * x[q];
    }
    stv<W>(Dinv, i, di);
    stv<W>(d1, i, d);
  }
  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&sum)[2], Con &,
                                    AT &) const {
    const double zw = src.ldw(W_ZW, v.zw, ci), sw = src.ldw(W_SW, v.sw, ci);
    const double tw = src.ldw(W_TW, v.tw, ci);
    const double zsw = src.ldw(W_ZSW, v.zsw, ci), ztw = src.ldw(W_ZTW, v.ztw, ci);
    Cw[ci] = pcu_rcp((pcu_div(sw, zsw) + pcu_div(tw, ztw)) + sum[0]);
    const double bzw = -(((wconst_at(k, ci) + sum[1]) - sw) + tw);
    const double bsw = (zsw - gamma_sw(k, ci)) - zw;
    const double btw = (ztw - k.gamma) + zw;
    const double bzsw = mu - sw * zsw;
    const double bztw = mu - tw * ztw;
    d2[ci] = bzw + pcu_div(bzsw + sw * bsw, zsw) - pcu_div(bztw + tw * btw, ztw);
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void C(const S &, long long, const double (&)[W],
                                    const Elem (&)[W], const Con &, AT &) const {}
};
struct DiagRhsF : DiagRhsFT<0> {};
struct DiagRhsHF : DiagRhsFT<1> {};

// ============================================================== MehrotraCorrF
// addMehrotraCorrectorResidual (IP.cpp:1729-1789): second-order terms of the
// affine predictor step added to the complementarity residuals.
// Traffic: reads 7N + 6W, writes 2N + 2W.
struct MehrotraCorrF : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  DVars p, r;  // step (read), residual (updated in place)
  const double *lb, *ub;
  IPConst k;

  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *) const {}
  __device__ __forceinline__ void B(long long ci, const double (&)[1], Con &,
                                    AccT &) const {
    r.zsw[ci] -= p.sw[ci] * p.zsw[ci];
    r.ztw[ci] -= p.tw[ci] * p.ztw[ci];
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
    double px[W], l[W], u[W], pz[W], rz[W];
    ldv<W>(p.x, i, px);
    if (k.use_lower) {
      ldv<W>(lb, i, l);
      ldv<W>(p.zl, i, pz);
      ldv<W>(r.zl, i, rz);
#pragma unroll
      for (int q = 0; q < W; q++)
        if (l[q] > -k.mbv) rz[q] -= px[q] * pz[q];
      stv<W>(r.zl, i, rz);
    }
    if (k.use_upper) {
      ldv<W>(ub, i, u);
      ldv<W>(p.zu, i, pz);
      ldv<W>(r.zu, i, rz);
#pragma unroll
      for (int q = 0; q < W; q++)
        if (u[q] < k.mbv) rz[q] += px[q] * pz[q];
      stv<W>(r.zu, i, rz);
    }
  }
};

// ============================================================== Pass1F
// First half of solveKKTDiagSystem (IP.cpp:2091-2139): d1, d2 and the first
// ParOptQuasiDefBlockMat::apply (SM.cpp:160-190), t1 = D0^-1 (d1, d2)|x.
// Traffic: reads 7N + 10W, writes 2N + W.
struct Pass1F : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // yw
  struct Elem {
    double d1, dinv;
  };
  DVars v, b;
  const double *lb, *ub, *Dinv, *Cw;
  double *d1, *d2, *t1;
  IPConst k;
  // every part of the right-hand side except b.x is scaled by bs: the alpha-scaled
  // variant of the solve that the GMRES path uses (IP.cpp:2441-2614); 1 otherwise
  double bs = 1.0;

  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1], AccT *acc) const {
    double x[W], l[W], u[W], bx[W], bzl[W], bzu[W], di[W], d[W];
    ldv<W>(v.x, i, x);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(b.x, i, bx);
    ldv<W>(Dinv, i, di);
#pragma unroll
    for (int q = 0; q < W; q++) bzl[q] = bzu[q] = 0.0;
    if (k.use_lower) ldv<W>(b.zl, i, bzl);
    if (k.use_upper) ldv<W>(b.zu, i, bzu);
#pragma unroll
    for (int q = 0; q < W; q++) {
      double t = bx[q];
      if (k.use_lower && l[q] > -k.mbv) t += bs * bzl[q] / (x[q] - l[q]);
      if (k.use_upper && u[q] < k.mbv) t -= bs * bzu[q] / (u[q] - x[q]);
      d[q] = t;
      e[q].d1 = t;
      e[q].dinv = di[q];
      part[q][0] = coef[q] * di[q] * t;
    }
    stv<W>(d1, i, d);
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1],
                                    Con &con, AccT &) const {
    const double sw = v.sw[ci], tw = v.tw[ci], zsw = v.zsw[ci], ztw = v.ztw[ci];
    const double dd = bs * (b.zw[ci] + (b.zsw[ci] + sw * b.sw[ci]) / zsw -
                            (b.ztw[ci] + tw * b.tw[ci]) / ztw);
    con.d[0] = Cw[ci] * (dd - sum[0]);
    d2[ci] = dd;
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AccT &) const {
    double t[W];
#pragma unroll
    for (int q = 0; q < W; q++) t[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
    stv<W>(t1, i, t);
  }
};

// ============================================================== Pass2F
// Second half of solveKKTDiagSystem (IP.cpp:2165-2242) merged with the
// Sherman-Morrison-Woodbury correction of computeKKTStep (IP.cpp:2716-2735):
//   d1' = d1 + sum_j alpha_j V_j,  V = [A | Z]   (alpha from the small dense
//   solves), (px, pzw) = D0^-1 (d1', d2), then the bound / slack multipliers.
// accumulate != 0 adds the result to the step (update.add(refine), IP.cpp:4990).
// Traffic: reads (9 + c + q)N + 10W, writes 3N + 5W (+3N + 5W reads when
// accumulating).
struct Pass2F : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // yw
  struct Elem {
    double d1, dinv;
  };
  DVars v, b, y;
  const double *lb, *ub, *Dinv, *Cw, *d1, *d2;
  ColTable V;
  CoefTable alpha;
  int ncols;
  int accumulate;
  IPConst k;
  double bs = 1.0;  // scale of the right-hand side parts (see Pass1F)

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(d1); p_(Dinv); p_(v.x); p_(lb); p_(ub);
    if (k.use_lower) { p_(v.zl); p_(b.zl); }
    if (k.use_upper) { p_(v.zu); p_(b.zu); }
    for (int j = 0; j < ncols; j++) p_(V.p[j]);
    if (accumulate) {
      p_(y.x);
      if (k.use_lower) p_(y.zl);
      if (k.use_upper) p_(y.zu);
    }
  }

  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1], AccT *acc) const {
    double d[W], di[W];
    ldv<W>(d1, i, d);
    ldv<W>(Dinv, i, di);
    for (int j = 0; j < ncols; j++) {
      double c[W];
      ldv<W>(V.p[j], i, c);
#pragma unroll
      for (int q = 0; q < W; q++) d[q] = fma(alpha.v[j], c[q], d[q]);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      e[q].d1 = d[q];
      e[q].dinv = di[q];
      part[q][0] = coef[q] * di[q] * d[q];
    }
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1],
                                    Con &con, AccT &) const {
    const double yw = Cw[ci] * (d2[ci] - sum[0]);
    con.d[0] = yw;
    const double sw = v.sw[ci], tw = v.tw[ci], zsw = v.zsw[ci], ztw = v.ztw[ci];
    const double pzsw = yw - bs * b.sw[ci];
    const double pztw = -bs * b.tw[ci] - yw;
    const double psw = (bs * b.zsw[ci] - sw * pzsw) / zsw;
    const double ptw = (bs * b.ztw[ci] - tw * pztw) / ztw;
    if (accumulate) {
      y.zw[ci] += yw;
      y.zsw[ci] += pzsw;
      y.ztw[ci] += pztw;
      y.sw[ci] += psw;
      y.tw[ci] += ptw;
    } else {
      y.zw[ci] = yw;
      y.zsw[ci] = pzsw;
      y.ztw[ci] = pztw;
      y.sw[ci] = psw;
      y.tw[ci] = ptw;
    }
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AccT &) const {
    double x[W], l[W], u[W], zl[W], zu[W], bzl[W], bzu[W];
    double px[W], pzl[W], pzu[W];
    ldv<W>(v.x, i, x);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = bzl[q] = bzu[q] = 0.0;
    if (k.use_lower) {
      ldv<W>(v.zl, i, zl);
      ldv<W>(b.zl, i, bzl);
    }
    if (k.use_upper) {
      ldv<W>(v.zu, i, zu);
      ldv<W>(b.zu, i, bzu);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      px[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
      pzl[q] = 0.0;
      pzu[q] = 0.0;
      if (k.use_lower && l[q] > -k.mbv)
        pzl[q] = (bs * bzl[q] - zl[q] * px[q]) / (x[q] - l[q]);
      if (k.use_upper && u[q] < k.mbv)
        pzu[q] = (bs * bzu[q] + zu[q] * px[q]) / (u[q] - x[q]);
    }
    if (accumulate) {
      double o[W];
      ldv<W>(y.x, i, o);
#pragma unroll
      for (int q = 0; q < W; q++) px[q] += o[q];
      if (k.use_lower) {
        ldv<W>(y.zl, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzl[q] += o[q];
      }
      if (k.use_upper) {
        ldv<W>(y.zu, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzu[q] += o[q];
      }
    }
    stv<W>(y.x, i, px);
    if (k.use_lower) stv<W>(y.zl, i, pzl);
    if (k.use_upper) stv<W>(y.zu, i, pzu);
  }
};

// Element / constraint terms of the step statistics, shared by StatsF and by
// Pass2SF (which produces the step in the same pass).
template <int W, class AccT_>
__device__ __forceinline__ void stats_elements(
    const IPConst &k, double tau, const double (&x)[W], const double (&l)[W],
    const double (&u)[W], const double (&zl)[W], const double (&zu)[W],
    const double (&px)[W], const double (&pzl)[W], const double (&pzu)[W],
    const double (&gv)[W], AccT_ &a) {
    double facs[W];  // product of the barrier arguments of each element
#pragma unroll
    for (int q = 0; q < W; q++) {
      const double dl = x[q] - l[q], du = u[q] - x[q];
      const double pxq = px[q];
      double fac = 1.0;
      const bool ml = k.use_lower && l[q] > -k.mbv;
      const bool mu_ = k.use_upper && u[q] < k.mbv;
      // Fraction to the boundary (IP.cpp:2959-2982, 3064-3091): the quotient is
      // only formed for elements that can lower the running minimum (the
      // product test keeps a 1e-12 slack so no candidate is lost).
      if (k.use_lower) {
        if (pxq < 0.0 && tau * dl <= -a.m[0] * pxq * (1.0 + 1e-12))
          a.m[0] = fmin(a.m[0], -tau * dl / pxq);
        if (pzl[q] < 0.0 && tau * zl[q] <= -a.m[1] * pzl[q] * (1.0 + 1e-12))
          a.m[1] = fmin(a.m[1], -tau * zl[q] / pzl[q]);
      }
      if (k.use_upper) {
        if (pxq > 0.0 && tau * du <= a.m[0] * pxq * (1.0 + 1e-12))
          a.m[0] = fmin(a.m[0], tau * du / pxq);
        if (pzu[q] < 0.0 && tau * zu[q] <= -a.m[1] * pzu[q] * (1.0 + 1e-12))
          a.m[1] = fmin(a.m[1], -tau * zu[q] / pzu[q]);
      }
      if (ml) {
        a.s[0] = fma(zl[q], dl, a.s[0]);
        a.s[1] = fma(zl[q], pxq, a.s[1]);
        a.s[2] = fma(pzl[q], dl, a.s[2]);
        a.s[3] = fma(pzl[q], pxq, a.s[3]);
      }
      if (mu_) {
        a.s[0] = fma(zu[q], du, a.s[0]);
        a.s[1] = fma(-zu[q], pxq, a.s[1]);
        a.s[2] = fma(pzu[q], du, a.s[2]);
        a.s[3] = fma(-pzu[q], pxq, a.s[3]);
      }
      // Barrier terms (IP.cpp:3684-3722).  The logarithms are accumulated as a
      // running product (lp_mul: slots 8, 9 hold mantissa product and exponent
      // sum; finalize() turns them into the sum of logs, so the reference's
      // > 1 / <= 1 buckets collapse into slot 8); with both bounds present the
      // two quotients share one reciprocal.
      if (ml && mu_) {
        const double prod = dl * du;
        fac *= prod;
        const double rinv = pcu_rcp(prod);
        const double rl = pxq * du * rinv, ru = pxq * dl * rinv;
        if (pxq > 0.0) {
          a.s[10] += rl;
          a.s[11] -= ru;
        } else {
          a.s[11] += rl;
          a.s[10] -= ru;
        }
      } else {
        if (ml) {
          fac *= dl;
          const double r = pcu_div(pxq, dl);
          if (pxq > 0.0) a.s[10] += r; else a.s[11] += r;
        }
        if (mu_) {
          fac *= du;
          const double r = pcu_div(pxq, du);
          if (pxq > 0.0) a.s[11] -= r; else a.s[10] -= r;
        }
      }
      a.s[16] = fma(gv[q], pxq, a.s[16]);
      a.s[17] = fma(pxq, pxq, a.s[17]);
      a.x[0] = fmax(a.x[0], fabs(pxq));
      facs[q] = fac;
    }
    if (W == 2) lp_mul2(a.s[8], a.s[9], facs[0], facs[W - 1]);
    else lp_mul(a.s[8], a.s[9], facs[0]);
}
template <class AccT_>
__device__ __forceinline__ void stats_constraint_vals(
    const IPConst &k, double tau, long long ci, double sw, double tw, double zsw,
    double ztw, double psw, double ptw, double pzsw, double pztw,
    const double (&sum)[2], AccT_ &acc) {
    // as in stats_elements: the quotient is only formed for a candidate that can
    // lower the running minimum (1e-12 slack: no candidate is lost)
    if (psw < 0.0 && tau * sw <= -acc.m[0] * psw * (1.0 + 1e-12))
      acc.m[0] = fmin(acc.m[0], -tau * sw / psw);
    if (ptw < 0.0 && tau * tw <= -acc.m[0] * ptw * (1.0 + 1e-12))
      acc.m[0] = fmin(acc.m[0], -tau * tw / ptw);
    if (pzsw < 0.0 && tau * zsw <= -acc.m[1] * pzsw * (1.0 + 1e-12))
      acc.m[1] = fmin(acc.m[1], -tau * zsw / pzsw);
    if (pztw < 0.0 && tau * ztw <= -acc.m[1] * pztw * (1.0 + 1e-12))
      acc.m[1] = fmin(acc.m[1], -tau * ztw / pztw);
    acc.s[4] += sw * zsw + tw * ztw;
    acc.s[5] += psw * zsw + ptw * ztw;
    acc.s[6] += sw * pzsw + tw * pztw;
    acc.s[7] += psw * pzsw + ptw * pztw;
    const double swtw = sw * tw;
    lp_mul(acc.s[12], acc.s[13], swtw);
    const double rinv = pcu_rcp(swtw);
    const double rs = psw * tw * rinv, rt = ptw * sw * rinv;
    if (psw > 0.0) acc.s[14] += rs; else acc.s[15] += rs;
    if (ptw > 0.0) acc.s[14] += rt; else acc.s[15] += rt;
    const double gsw = gamma_sw(k, ci), gtw = k.gamma;
    acc.s[18] += gsw * sw + gtw * tw;
    acc.s[19] += gsw * psw + gtw * ptw;
    const double rw1 = ((wconst_at(k, ci) + sum[0]) - sw) + tw;
    const double rw2 = (sum[1] - psw) + ptw;
    acc.s[20] = fma(rw1, rw1, acc.s[20]);
    acc.s[21] = fma(rw1, rw2, acc.s[21]);
}
template <class AccT_>
__device__ __forceinline__ void stats_constraint(const IPConst &k, double tau,
                                                 long long ci, const DVars &v,
                                                 const DVars &p,
                                                 const double (&sum)[2],
                                                 AccT_ &acc) {
    stats_constraint_vals(k, tau, ci, v.sw[ci], v.tw[ci], v.zsw[ci], v.ztw[ci], p.sw[ci],
                          p.tw[ci], p.zsw[ci], p.ztw[ci], sum, acc);
}

// ============================================================== StatsF
// One pass giving every reduction needed between the KKT step and the line
// search: computeMaxStep (IP.cpp:2942-3103), computeCompStep (IP.cpp:2825-2923,
// as the 4 coefficients of its bilinear form in (alpha_x, alpha_z)), and the
// sums of evalMeritInitDeriv / evalInfeasDeriv (IP.cpp:3652-3790, 3465-3509).
// Traffic: reads 9N + 8W.
//   sums: 0-3 bound comp poly [1, ax, az, ax*az]; 4-7 sparse comp poly;
//         8,9 pos/neg log (bounds); 10,11 pos/neg p/(.) (bounds);
//         12,13 pos/neg log (sw,tw); 14,15 pos/neg p/(.) (sw,tw);
//         16 g.p; 17 p.p; 18 gam.(sw,tw); 19 gam.(psw,ptw);
//         20 |cw - sw + tw|^2; 21 (cw - sw + tw).(Aw p - psw + ptw)
//   maxima: 0 |px|_inf;  mins: 0 max_x, 1 max_z
struct StatsF : NoStreams {
  static constexpr int MINB = PCU_MINB_STATS;
  static constexpr int NS = 22, NX = 1, NM = 2, NB = 2;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  DVars v, p;
  const double *lb, *ub, *g;
  double tau;
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(p.x); p_(lb); p_(ub); p_(g);
    if (k.use_lower) { p_(v.zl); p_(p.zl); }
    if (k.use_upper) { p_(v.zu); p_(p.zu); }
  }

  // All element reductions happen here (acc is null on the generic path's
  // first, sum-only visit of an element).
  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W],
                                    Elem (&)[W], double (&part)[W][2],
                                    AccT *acc) const {
    double x[W], l[W], u[W], px[W];
    ldv<W>(v.x, i, x);
    ldv<W>(p.x, i, px);
#pragma unroll
    for (int q = 0; q < W; q++) {
      part[q][0] = coef[q] * x[q];
      part[q][1] = coef[q] * px[q];
    }
    if (!acc) return;
    double zl[W], zu[W], pzl[W], pzu[W], gv[W];
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = pzl[q] = pzu[q] = 0.0;
    if (k.use_lower) {
      ldv<W>(v.zl, i, zl);
      ldv<W>(p.zl, i, pzl);
    }
    if (k.use_upper) {
      ldv<W>(v.zu, i, zu);
      ldv<W>(p.zu, i, pzu);
    }
    stats_elements<W>(k, tau, x, l, u, zl, zu, px, pzl, pzu, gv, *acc);
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[2], Con &,
                                    AccT &acc) const {
    stats_constraint(k, tau, ci, v, p, sum, acc);
  }
  template <int W>
  __device__ __forceinline__ void C(long long, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {}
  __device__ __forceinline__ void finalize(AccT &acc) const {
    acc.s[8] = lp_value(acc.s[8], acc.s[9]);
    acc.s[9] = 0.0;
    acc.s[12] = lp_value(acc.s[12], acc.s[13]);
    acc.s[13] = 0.0;
  }
};

// ============================================================== Pass2SF
// Pass2F (the last pass of the iteration's KKT solves) fused with StatsF: the
// step statistics are taken from the step while it is still in registers, so
// the separate 9N + 8W statistics pass disappears (one extra stream: g).
// Traffic: Pass2F + N.   Reductions: as StatsF (sums in shared memory).
//
// Pass2SVF (FV = 1): the same pass as the ONLY pass of a KKT solve whose right-hand
// side is the residual of the variables, computeKKTRes(vars, mu_rhs) (the default
// iteration, refined in the column space of [A|Z]: pcu_dense_solve).  The bound rows
// (IP.cpp:1417-1444) and the weighting rows (IP.cpp:1361-1389) of that residual are
// formed from the variables instead of being read; never accumulating.
// Traffic: reads (8 + m)N + 7W, writes 3N + 5W (+ N: A p_z).
//
// Pass2SVHF (FV = 1, HD = 1; use_diag_hessian): also reads h and adds one sum,
// s[22] = sum h p^2, the curvature term of the merit derivative (p^T B p with
// B = diag(h)).  h is read, not recovered from Dinv: 1/Dinv - sigma - bound terms
// cancels where the bound terms dominate.  Reads (9 + m)N + 7W.
struct ConP2S {  // yw broadcast; the leader lane keeps the constraint's values for E
  static constexpr int ND = 1;
  double d[1];
  double sw, tw, zsw, ztw, psw, ptw, pzsw, pztw;
  __device__ __forceinline__ void zero() { d[0] = 0.0; }
};
// mu_rhs (the barrier of the right-hand side) exists in Pass2SVF only: an empty base in
// Pass2SF keeps that kernel's parameter block, and with it ptxas's code, unchanged
template <int FV> struct Pass2SFRhs { double mu_rhs; };
template <> struct Pass2SFRhs<0> {};
template <int FV, int HD = 0>
struct Pass2SFT : NoStreams, Pass2SFRhs<FV>, HessDiagPtr<HD> {
  static_assert(FV || !HD, "the diagonal Hessian runs on the variables' right-hand side");
  static constexpr int SRC = 1;
  // Pass2SF follows Pass2R1F (upwards); Pass2SVF follows the Gram pass (downwards)
  static constexpr int REVERSE = FV ? 0 : 1;
  static constexpr int MINB = PCU_MINB_PASS2S;
  static constexpr int NS = 22 + HD, NX = 1, NM = 2, NB = 1, NB2 = 2;
  static constexpr int SMEM = NS * PCU_TILE_THREADS * 8;
  typedef AccS<NS, NX, NM> AccT;
  typedef ConP2S Con;
  struct Elem {
    double d1, dinv;
  };
  // staged slots (tma_tile_kernel): N-streams, then the columns; W-streams
  enum { S_D1, S_DINV, S_X, S_LB, S_UB, S_G, S_ZL, S_BZL, S_ZU, S_BZU, S_YX, S_YZL, S_YZU, S_H };
  static constexpr int S_V0 = S_H + HD;
  static constexpr int NFIX = S_V0;  // fixed slots; the columns follow
  enum { W_CW, W_D2, W_SW, W_TW, W_ZSW, W_ZTW, W_BSW, W_BTW, W_BZSW, W_BZTW,
         W_YZW, W_YZSW, W_YZTW, W_YSW, W_YTW, NWSLOTS };
  static constexpr int W_ZW = W_BSW;  // FV: zw takes the slot of the unread b.sw
  DVars v, b, y;
  const double *lb, *ub, *Dinv, *Cw, *d1, *d2, *g;
  ColTable V;
  CoefTable alpha;
  int cbank;  // >= 0: alpha at this offset of the constant bank (chain mode); -1: `alpha`
  int ncols;
  int accumulate;  // FV: 0
  double tau;
  IPConst k;
  // optional output: sum over the first nca columns (the constraint gradients) of
  // alpha_j V_j = A p_z of this solve; the update pass then forms -(g - A z+) from
  // g - A z (left by the previous update pass) without re-reading the nca columns
  double *apz = nullptr;
  int nca = 0;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(d1); p_(Dinv); p_(v.x); p_(lb); p_(ub); p_(g);
    if (k.use_lower) { p_(v.zl); if (!FV) p_(b.zl); }
    if (k.use_upper) { p_(v.zu); if (!FV) p_(b.zu); }
    if constexpr (HD) p_(this->h);
    for (int j = 0; j < ncols; j++) p_(V.p[j]);
    if (!FV && accumulate) {
      p_(y.x);
      if (k.use_lower) p_(y.zl);
      if (k.use_upper) p_(y.zu);
    }
  }
  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_D1, d1); p_.n(S_DINV, Dinv); p_.n(S_X, v.x); p_.n(S_LB, lb); p_.n(S_UB, ub);
    p_.n(S_G, g);
    if (k.use_lower) { p_.n(S_ZL, v.zl); if (!FV) p_.n(S_BZL, b.zl); }
    if (k.use_upper) { p_.n(S_ZU, v.zu); if (!FV) p_.n(S_BZU, b.zu); }
    if (!FV && accumulate) {
      p_.n(S_YX, y.x);
      if (k.use_lower) p_.n(S_YZL, y.zl);
      if (k.use_upper) p_.n(S_YZU, y.zu);
    }
    if constexpr (HD) p_.n(S_H, this->h);
    for (int j = 0; j < ncols; j++) p_.n(S_V0 + j, V.p[j]);
    p_.w(W_CW, Cw); p_.w(W_D2, d2);
    p_.w(W_SW, v.sw); p_.w(W_TW, v.tw); p_.w(W_ZSW, v.zsw); p_.w(W_ZTW, v.ztw);
    if (FV) {
      p_.w(W_ZW, v.zw);
    } else {
      p_.w(W_BSW, b.sw); p_.w(W_BTW, b.tw); p_.w(W_BZSW, b.zsw); p_.w(W_BZTW, b.ztw);
    }
    if (!FV && accumulate) {
      p_.w(W_YZW, y.zw); p_.w(W_YZSW, y.zsw); p_.w(W_YZTW, y.ztw);
      p_.w(W_YSW, y.sw); p_.w(W_YTW, y.tw);
    }
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void A(const S &src, long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1], AT *) const {
    double d[W], di[W], qa[W];
    src.template ld<W>(S_D1, d1, i, d);
    src.template ld<W>(S_DINV, Dinv, i, di);
#pragma unroll
    for (int q = 0; q < W; q++) qa[q] = 0.0;
    int j = 0;
    for (; j + 4 <= ncols; j += 4) {  // four columns per batch: loads first
      double c[4][W];
#pragma unroll
      for (int jj = 0; jj < 4; jj++) src.template ldc<W>(j + jj, V.p[j + jj], i, c[jj]);
      double al[4];
#pragma unroll
      for (int jj = 0; jj < 4; jj++) al[jj] = pcu_coef(cbank, alpha, j + jj);
#pragma unroll
      for (int jj = 0; jj < 4; jj++) {
#pragma unroll
        for (int q = 0; q < W; q++) d[q] = fma(al[jj], c[jj][q], d[q]);
        if (apz && j + jj < nca) {
#pragma unroll
          for (int q = 0; q < W; q++) qa[q] = fma(al[jj], c[jj][q], qa[q]);
        }
      }
    }
    for (; j < ncols; j++) {
      double c[W];
      src.template ldc<W>(j, V.p[j], i, c);
      const double aj = pcu_coef(cbank, alpha, j);
#pragma unroll
      for (int q = 0; q < W; q++) d[q] = fma(aj, c[q], d[q]);
      if (apz && j < nca) {
#pragma unroll
        for (int q = 0; q < W; q++) qa[q] = fma(aj, c[q], qa[q]);
      }
    }
    if (apz) stv<W>(apz, i, qa);
#pragma unroll
    for (int q = 0; q < W; q++) {
      e[q].d1 = d[q];
      e[q].dinv = di[q];
      part[q][0] = coef[q] * di[q] * d[q];
    }
  }
  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&sum)[1],
                                    Con &con, AT &) const {
    const double yw = src.ldw(W_CW, Cw, ci) * (src.ldw(W_D2, d2, ci) - sum[0]);
    con.d[0] = yw;
    const double sw = src.ldw(W_SW, v.sw, ci), tw = src.ldw(W_TW, v.tw, ci);
    const double zsw = src.ldw(W_ZSW, v.zsw, ci), ztw = src.ldw(W_ZTW, v.ztw, ci);
    double bsw, btw, bzsw, bztw;
    if constexpr (FV) {  // IP.cpp:1361-1389
      const double zw = src.ldw(W_ZW, v.zw, ci);
      bsw = (zsw - gamma_sw(k, ci)) - zw;
      btw = (ztw - k.gamma) + zw;
      bzsw = this->mu_rhs - sw * zsw;
      bztw = this->mu_rhs - tw * ztw;
    } else {
      bsw = src.ldw(W_BSW, b.sw, ci);
      btw = src.ldw(W_BTW, b.tw, ci);
      bzsw = src.ldw(W_BZSW, b.zsw, ci);
      bztw = src.ldw(W_BZTW, b.ztw, ci);
    }
    double pzsw = yw - bsw;
    double pztw = -btw - yw;
    double psw = pcu_div(bzsw - sw * pzsw, zsw);
    double ptw = pcu_div(bztw - tw * pztw, ztw);
    double pzw = yw;
    if (!FV && accumulate) {
      pzw = src.ldw(W_YZW, y.zw, ci) + yw;
      pzsw = src.ldw(W_YZSW, y.zsw, ci) + pzsw;
      pztw = src.ldw(W_YZTW, y.ztw, ci) + pztw;
      psw = src.ldw(W_YSW, y.sw, ci) + psw;
      ptw = src.ldw(W_YTW, y.tw, ci) + ptw;
    }
    y.zw[ci] = pzw;
    y.zsw[ci] = pzsw;
    y.ztw[ci] = pztw;
    y.sw[ci] = psw;
    y.tw[ci] = ptw;
    con.sw = sw; con.tw = tw; con.zsw = zsw; con.ztw = ztw;
    con.psw = psw; con.ptw = ptw; con.pzsw = pzsw; con.pztw = pztw;
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void C2(const S &src, long long i, const double (&coef)[W],
                                     const Elem (&e)[W], const Con &con, AT &acc,
                                     double (&part2)[W][2]) const {
    double x[W], l[W], u[W], zl[W], zu[W], bzl[W], bzu[W], gv[W];
    double px[W], pzl[W], pzu[W];
    src.template ld<W>(S_X, v.x, i, x);
    src.template ld<W>(S_LB, lb, i, l);
    src.template ld<W>(S_UB, ub, i, u);
    src.template ld<W>(S_G, g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = bzl[q] = bzu[q] = 0.0;
    if (k.use_lower) {
      src.template ld<W>(S_ZL, v.zl, i, zl);
      if (!FV) src.template ld<W>(S_BZL, b.zl, i, bzl);
    }
    if (k.use_upper) {
      src.template ld<W>(S_ZU, v.zu, i, zu);
      if (!FV) src.template ld<W>(S_BZU, b.zu, i, bzu);
    }
    if constexpr (FV) {  // rzl, rzu of computeKKTRes (IP.cpp:1417-1444)
#pragma unroll
      for (int q = 0; q < W; q++) {
        bzl[q] = -((x[q] - l[q]) * zl[q] - k.kappa * this->mu_rhs);
        bzu[q] = -((u[q] - x[q]) * zu[q] - k.kappa * this->mu_rhs);
      }
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      px[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
      pzl[q] = 0.0;
      pzu[q] = 0.0;
      if (k.use_lower && l[q] > -k.mbv)
        pzl[q] = pcu_div(bzl[q] - zl[q] * px[q], x[q] - l[q]);
      if (k.use_upper && u[q] < k.mbv)
        pzu[q] = pcu_div(bzu[q] + zu[q] * px[q], u[q] - x[q]);
    }
    if (!FV && accumulate) {
      double o[W];
      src.template ld<W>(S_YX, y.x, i, o);
#pragma unroll
      for (int q = 0; q < W; q++) px[q] += o[q];
      if (k.use_lower) {
        src.template ld<W>(S_YZL, y.zl, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzl[q] += o[q];
      }
      if (k.use_upper) {
        src.template ld<W>(S_YZU, y.zu, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzu[q] += o[q];
      }
    }
    stv<W>(y.x, i, px);
    if (k.use_lower) stv<W>(y.zl, i, pzl);
    if (k.use_upper) stv<W>(y.zu, i, pzu);
    stats_elements<W>(k, tau, x, l, u, zl, zu, px, pzl, pzu, gv, acc);
    if constexpr (HD) {
      double hv[W];
      src.template ld<W>(S_H, this->h, i, hv);
#pragma unroll
      for (int q = 0; q < W; q++) acc.s[22] = fma(hv[q] * px[q], px[q], acc.s[22]);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      part2[q][0] = coef[q] * x[q];
      part2[q][1] = coef[q] * px[q];
    }
  }
  template <class S, class AT>
  __device__ __forceinline__ void E(const S &, long long ci, const double (&sum2)[2],
                                    const Con &con, AT &acc) const {
    stats_constraint_vals(k, tau, ci, con.sw, con.tw, con.zsw, con.ztw, con.psw, con.ptw,
                          con.pzsw, con.pztw, sum2, acc);
  }
  template <class AT>
  __device__ __forceinline__ void finalize(AT &acc) const {
    acc.s[8] = lp_value(acc.s[8], acc.s[9]);
    acc.s[9] = 0.0;
    acc.s[12] = lp_value(acc.s[12], acc.s[13]);
    acc.s[13] = 0.0;
  }
};
// distinct types, so that kernel names and profiles tell the two passes apart
struct Pass2SF : Pass2SFT<0> {};
struct Pass2SVF : Pass2SFT<1> {};
struct Pass2SVHF : Pass2SFT<1, 1> {};

// The merit terms of a trial point, shared by TrialF and TrialUpdateF so that both
// take them with the same expressions.  Slots from `o`: o, o+1 running product of the
// bound barrier factors; o+2, o+3 that of sw tw; o+4 gam.(sw, tw); o+5 |cw - sw + tw|^2.
// Barrier factor of one element at the trial point r.
__device__ __forceinline__ double trial_bound_factor(const IPConst &k, double r, double l,
                                                     double u) {
  const bool ml = k.use_lower && l > -k.mbv;
  const bool mu_ = k.use_upper && u < k.mbv;
  const double dl = r - l, du = u - r;
  return (ml ? dl : 1.0) * (mu_ ? du : 1.0);
}
template <int W, class AT>
__device__ __forceinline__ void trial_bound_logs(int o, const double (&f)[W], AT &acc) {
  if (W == 2) lp_mul2(acc.s[o], acc.s[o + 1], f[0], f[W - 1]);
  else lp_mul(acc.s[o], acc.s[o + 1], f[0]);
}
// sw, tw: the trial slacks; sum0: the constraint's block sum of the trial point
template <class AT>
__device__ __forceinline__ void trial_constraint(int o, const IPConst &k, long long ci,
                                                 double sw, double tw, double sum0,
                                                 AT &acc) {
  lp_mul(acc.s[o + 2], acc.s[o + 3], sw * tw);
  acc.s[o + 4] += gamma_sw(k, ci) * sw + k.gamma * tw;
  const double rw = ((wconst_at(k, ci) + sum0) - sw) + tw;
  acc.s[o + 5] = fma(rw, rw, acc.s[o + 5]);
}
template <class AT>
__device__ __forceinline__ void trial_finalize(int o, AT &acc) {
  acc.s[o] = lp_value(acc.s[o], acc.s[o + 1]);
  acc.s[o + 1] = 0.0;
  acc.s[o + 2] = lp_value(acc.s[o + 2], acc.s[o + 3]);
  acc.s[o + 3] = 0.0;
}

// ============================================================== TrialF
// Line-search trial point (IP.cpp:3997-4013: rx, rsw, rtw via computeStepVec)
// fused with the reductions of evalMeritFunc / evalInfeas (IP.cpp:3524-3601,
// 3438-3460) at that point.  ax = alpha * alpha_x (the step is kept unscaled).
// Traffic: reads 4N + 4W, writes N + 2W.
//   sums: 0,1 pos/neg log (bounds); 2,3 pos/neg log (sw,tw); 4 gam.(rsw,rtw);
//         5 |cw(rx) - rsw + rtw|^2
struct TrialF : NoStreams {
  static constexpr int SRC = 1;
  static constexpr int NS = 6, NX = 0, NM = 0, NB = 1;
  enum { S_X, S_PX, S_LB, S_UB, NSLOTS };
  static constexpr int NFIX = NSLOTS;  // fixed slots; the columns follow
  static constexpr int TROWS = 1024;
  enum { W_SW, W_TW, W_PSW, W_PTW, NWSLOTS };
  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_X, v.x); p_.n(S_PX, p.x); p_.n(S_LB, lb); p_.n(S_UB, ub);
    p_.w(W_SW, v.sw); p_.w(W_TW, v.tw); p_.w(W_PSW, p.sw); p_.w(W_PTW, p.tw);
  }
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {
    double f;
  };
  DVars v, p;
  const double *lb, *ub;
  double *rx, *rsw, *rtw;
  double ax;
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(p.x); p_(lb); p_(ub);
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void A(const S &src, long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1], AT *acc) const {
    double x[W], l[W], u[W], px[W], r[W];
    src.template ld<W>(S_X, v.x, i, x);
    src.template ld<W>(S_LB, lb, i, l);
    src.template ld<W>(S_UB, ub, i, u);
    src.template ld<W>(S_PX, p.x, i, px);
#pragma unroll
    for (int q = 0; q < W; q++) {
      r[q] = step_clip(x[q], ax, px[q], l[q], u[q], k.dp);
      // factor of the running product whose logarithm is the barrier sum
      e[q].f = trial_bound_factor(k, r[q], l[q], u[q]);
      part[q][0] = coef[q] * r[q];
    }
    stv<W>(rx, i, r);
  }
  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&sum)[1], Con &,
                                    AT &acc) const {
    const double s = step_clip0(src.ldw(W_SW, v.sw, ci), ax, src.ldw(W_PSW, p.sw, ci), k.dp);
    const double t = step_clip0(src.ldw(W_TW, v.tw, ci), ax, src.ldw(W_PTW, p.tw, ci), k.dp);
    rsw[ci] = s;
    rtw[ci] = t;
    trial_constraint(0, k, ci, s, t, sum[0], acc);
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void C(const S &, long long, const double (&)[W],
                                    const Elem (&e)[W], const Con &,
                                    AT &acc) const {
    double f[W];
#pragma unroll
    for (int q = 0; q < W; q++) f[q] = e[q].f;
    trial_bound_logs<W>(0, f, acc);
  }
  template <class AT>
  __device__ __forceinline__ void finalize(AT &acc) const {
    trial_finalize(0, acc);
  }
};

// ============================================================== Update1F
// computeStepAndUpdate, first half (IP.cpp:4178-4216): every variable takes its
// step (ax = alpha*alpha_x for primal, az = alpha*alpha_z for dual parts) and
// y_qn = -g + sum_j z_j A_j + Aw^T zw with the NEW multipliers and the OLD
// gradients.  Traffic: reads (6 + c)N + 10W, writes 4N + 5W.
// STATS = 1 also takes, at the NEW point, the part of the next iteration's residual
// statistics that does not depend on the new gradients (computeComp, IP.cpp:2742-2820;
// the sparse and bound parts of computeResNorm, IP.cpp:1588-1723) -- the values are in
// registers here anyway, and together with Update2F's |rx| the stand-alone residual
// pass (ResF) of a default iteration disappears.  Same expressions, same accumulation
// order as ResF.   sums: 0 bound comp product, 1 comp count, 2 sparse comp product;
// maxima: 0 |rzw|, 1 |rsw| / |rtw|, 2 bound products, 3 sparse products; minima: 0
// bound products, 1 sparse products.
// TRIAL = 1 (TrialUpdateF) runs BEFORE the objective callback as the line search's
// first trial: the new point goes to r (r.x = rx, r.sw = rsw, r.tw = rtw: the trial
// point TrialF would have written, bit for bit) instead of v, and the pass also takes
// TrialF's six merit sums at it, in slots 3-8 (TrialF's 0-5).  The host exchanges r
// with v when the trial is accepted -- one pass instead of TrialF + Update1FT.
// Traffic: the words of Update1FT (TrialF's 5N + 6W disappear); six more sums, and the
// merit terms' arithmetic on every element and constraint.
template <int TRIAL> struct Update1Out { DVars r; };
template <> struct Update1Out<0> {};
template <int STATS, int TRIAL = 0>
struct Update1FT : NoStreams, Update1Out<TRIAL> {
  static constexpr int SRC = 1;
  // from the last tile down: after TrialF, or with TRIAL after Pass2SVF, both of which
  // walk from the first tile up
  static constexpr int REVERSE = 1;
  // the merit sums do not fit the register-fed kernel's 73 registers without spills
  static constexpr int MINB = TRIAL ? 5 : NoStreams::MINB;
  static constexpr int TS = STATS ? 3 : 0;  // first slot of the merit sums (TRIAL)
  static constexpr int NS = TS + (TRIAL ? 6 : 0), NX = STATS ? 4 : 0,
                       NM = STATS ? 2 : 0, NB = (STATS || TRIAL) ? 1 : 0;
  enum { S_X, S_PX, S_LB, S_UB, S_ZL, S_PZL, S_ZU, S_PZU, S_G, S_A0 };
  static constexpr int NFIX = S_A0;  // fixed slots; the columns follow
  static constexpr int TROWS = 512;
  enum { W_ZW, W_SW, W_TW, W_ZSW, W_ZTW, W_PZW, W_PSW, W_PTW, W_PZSW, W_PZTW, NWSLOTS };
  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_X, v.x); p_.n(S_PX, p.x); p_.n(S_LB, lb); p_.n(S_UB, ub);
    if (k.use_lower) { p_.n(S_ZL, v.zl); p_.n(S_PZL, p.zl); }
    if (k.use_upper) { p_.n(S_ZU, v.zu); p_.n(S_PZU, p.zu); }
    if (yqn) {
      p_.n(S_G, g);
      for (int j = 0; j < ncon; j++) p_.n(S_A0 + j, Acol.p[j]);
    }
    p_.w(W_ZW, v.zw); p_.w(W_SW, v.sw); p_.w(W_TW, v.tw); p_.w(W_ZSW, v.zsw);
    p_.w(W_ZTW, v.ztw);
    p_.w(W_PZW, p.zw); p_.w(W_PSW, p.sw); p_.w(W_PTW, p.tw); p_.w(W_PZSW, p.zsw);
    p_.w(W_PZTW, p.ztw);
  }
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // new zw
  struct Elem {
    double x;  // the new x
  };
  DVars v, p;
  const double *lb, *ub, *g;
  ColTable Acol;
  CoefTable z;  // NEW dense multipliers
  int ncon;
  double *yqn;  // null when no quasi-Newton pair is formed
  double ax, az;
  IPConst k;

  __device__ __forceinline__ const DVars &out() const {  // where the new point goes
    if constexpr (TRIAL) return this->r;
    else return v;
  }

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(p.x); p_(lb); p_(ub);
    if (k.use_lower) { p_(v.zl); p_(p.zl); }
    if (k.use_upper) { p_(v.zu); p_(p.zu); }
    if (yqn) {
      p_(g);
      for (int j = 0; j < ncon; j++) p_(Acol.p[j]);
    }
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void A(const S &src, long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1], AT *) const {
    double x[W], l[W], u[W], px[W];
    src.template ld<W>(S_X, v.x, i, x);
    src.template ld<W>(S_LB, lb, i, l);
    src.template ld<W>(S_UB, ub, i, u);
    src.template ld<W>(S_PX, p.x, i, px);
#pragma unroll
    for (int q = 0; q < W; q++) {
      e[q].x = step_clip(x[q], ax, px[q], l[q], u[q], k.dp);
      part[q][0] = coef[q] * e[q].x;
    }
  }
  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&sum)[1], Con &con,
                                    AT &acc) const {
    const double zwn = fma(az, src.ldw(W_PZW, p.zw, ci), src.ldw(W_ZW, v.zw, ci));  // no clipping (IP.cpp:4181)
    con.d[0] = zwn;
    const double sw = step_clip0(src.ldw(W_SW, v.sw, ci), ax, src.ldw(W_PSW, p.sw, ci), k.dp);
    const double tw = step_clip0(src.ldw(W_TW, v.tw, ci), ax, src.ldw(W_PTW, p.tw, ci), k.dp);
    const double zsw = step_clip0(src.ldw(W_ZSW, v.zsw, ci), az, src.ldw(W_PZSW, p.zsw, ci), k.dp);
    const double ztw = step_clip0(src.ldw(W_ZTW, v.ztw, ci), az, src.ldw(W_PZTW, p.ztw, ci), k.dp);
    const DVars &o = out();
    o.zw[ci] = zwn;
    o.sw[ci] = sw;
    o.tw[ci] = tw;
    o.zsw[ci] = zsw;
    o.ztw[ci] = ztw;
    if (TRIAL) trial_constraint(TS, k, ci, sw, tw, sum[0], acc);  // TrialF::B
    if (STATS) {  // ResF::B at the new point
      const double gsw = gamma_sw(k, ci), gtw = k.gamma;
      const double rzw = -(((wconst_at(k, ci) + sum[0]) - sw) + tw);
      const double rsw = (zsw - gsw) - zwn;
      const double rtw = (ztw - gtw) + zwn;
      const double asw = sw * zsw, atw = tw * ztw;
      acc.x[3] = fmax(acc.x[3], fmax(asw, atw));
      acc.m[1] = fmin(acc.m[1], fmin(asw, atw));
      acc.s[2] += asw + atw;
      acc.s[1] += 2.0;
      acc.x[0] = fmax(acc.x[0], fabs(rzw));
      acc.x[1] = fmax(acc.x[1], fmax(fabs(rsw), fabs(rtw)));
    }
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void C(const S &src, long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AT &acc) const {
    double l[W], u[W], zl[W], zu[W], x[W];
#pragma unroll
    for (int q = 0; q < W; q++) {
      x[q] = e[q].x;
      zl[q] = zu[q] = 0.0;
    }
    if (STATS || TRIAL) {
      src.template ld<W>(S_LB, lb, i, l);
      src.template ld<W>(S_UB, ub, i, u);
    }
    const DVars &o = out();
    if (k.use_lower) {
      double pzl[W];
      src.template ld<W>(S_ZL, v.zl, i, zl);
      src.template ld<W>(S_PZL, p.zl, i, pzl);
#pragma unroll
      for (int q = 0; q < W; q++) zl[q] = step_clip0(zl[q], az, pzl[q], k.dp);
      stv<W>(o.zl, i, zl);
    }
    if (k.use_upper) {
      double pzu[W];
      src.template ld<W>(S_ZU, v.zu, i, zu);
      src.template ld<W>(S_PZU, p.zu, i, pzu);
#pragma unroll
      for (int q = 0; q < W; q++) zu[q] = step_clip0(zu[q], az, pzu[q], k.dp);
      stv<W>(o.zu, i, zu);
    }
    if (yqn) {
      double gv[W], yv[W];
      src.template ld<W>(S_G, g, i, gv);
#pragma unroll
      for (int q = 0; q < W; q++) yv[q] = -gv[q];
      for (int j = 0; j < ncon; j++) {
        double a[W];
        src.template ldc<W>(j, Acol.p[j], i, a);
#pragma unroll
        for (int q = 0; q < W; q++) yv[q] = fma(z.v[j], a[q], yv[q]);
      }
#pragma unroll
      for (int q = 0; q < W; q++) yv[q] = fma(coef[q], con.d[0], yv[q]);
      stv<W>(yqn, i, yv);
    }
    stv<W>(o.x, i, x);
    if (TRIAL) {  // TrialF::A / C: the barrier factors of the bounds
      double f[W];
#pragma unroll
      for (int q = 0; q < W; q++) f[q] = trial_bound_factor(k, x[q], l[q], u[q]);
      trial_bound_logs<W>(TS, f, acc);
    }
    if (STATS) {  // ResF::A / C at the new point: complementarity of the bounds
#pragma unroll
      for (int q = 0; q < W; q++) {
        const bool ml = k.use_lower && (l[q] > -k.mbv);
        const bool mu_ = k.use_upper && (u[q] < k.mbv);
        const double dl = x[q] - l[q], du = u[q] - x[q];
        double cp = 0.0, cc = 0.0, amax = 0.0, amin = 1.0e300;
        if (ml) {
          const double a = dl * zl[q];
          cp += a;
          cc += 1.0;
          amax = fmax(amax, a);
          amin = fmin(amin, a);
        }
        if (mu_) {
          const double a = du * zu[q];
          cp += a;
          cc += 1.0;
          amax = fmax(amax, a);
          amin = fmin(amin, a);
        }
        acc.s[0] += cp;
        acc.s[1] += cc;
        acc.x[2] = fmax(acc.x[2], amax);
        acc.m[0] = fmin(acc.m[0], amin);
      }
    }
  }
  template <class AT>
  __device__ __forceinline__ void finalize(AT &acc) const {
    if (TRIAL) trial_finalize(TS, acc);
  }
};
typedef Update1FT<0> Update1F;
// a distinct type, so that kernel names and profiles tell it from the stand-alone pass
struct TrialUpdateF : Update1FT<1, 1> {};

// ============================================================== Update2F
// computeStepAndUpdate, second half (IP.cpp:4244-4256) after the new gradients:
//   s_qn = ax * px,  y_qn += g - sum_j z_j A_j - Aw^T zw
// fused with the three dot products that open ParOptLBFGS::update /
// ParOptLSR1::update (QN.cpp:168-170, 641-642).
// Traffic: reads (3 + c)N + W, writes 2N.   sums: 0 y.y, 1 y.s, 2 s.s
// RX = 1 (+ 2N reads: zl, zu) also takes |rx|_inf of the NEXT iteration's residual
// rx = zl - zu - g + sum_j z_j A_j + Aw^T zw (computeKKTRes, IP.cpp:1337-1399, with
// ResF's expression order) -- see Update1FT<1>.   maxima: 0 |rx|
// TR: rows per staged tile -- 1024 for a handful of streams, 128 when the ncon columns make
// a 1024-row stage too large for the ring (C4: 105 streams)
template <int RX, int TR = 1024>
struct Update2FT : NoStreams {
  static constexpr int SRC = 1;
  static constexpr int REVERSE = 1;  // after the gradient callbacks (upwards); DiagRhsF follows upwards
  static constexpr int NS = 3, NX = RX ? 1 : 0, NM = 0, NB = 0;
  enum { S_Y, S_G, S_PX, S_ZL, S_ZU, S_A0 };
  static constexpr int NFIX = S_A0;  // fixed slots; the columns follow
  static constexpr int TROWS = TR;
  enum { W_ZW, NWSLOTS };
  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_Y, yqn); p_.n(S_G, g); p_.n(S_PX, px);
    if (RX) { p_.n(S_ZL, zl); p_.n(S_ZU, zu); }
    for (int j = 0; j < ncon; j++) p_.n(S_A0 + j, Acol.p[j]);
    p_.w(W_ZW, zw);
  }
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // zw
  struct Elem {};
  const double *zw, *px, *g;
  const double *zl, *zu;  // RX only; null when the bound is not used
  ColTable Acol;
  CoefTable z;
  int ncon;
  double *yqn, *sqn;
  double ax;
  // optional output: g - sum_j z_j A_j at the new point, the part of the next
  // iteration's residual rx that needs the constraint gradients (DiagRhsF then reads
  // this vector instead of g and the ncon columns)
  double *gaz = nullptr;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(yqn); p_(g); p_(px);
    if (RX) { p_(zl); p_(zu); }
    for (int j = 0; j < ncon; j++) p_(Acol.p[j]);
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void A(const S &, long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AT *) const {}
  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&)[1], Con &con,
                                    AT &) const {
    con.d[0] = src.ldw(W_ZW, zw, ci);
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void C(const S &src, long long i, const double (&coef)[W],
                                    const Elem (&)[W], const Con &con,
                                    AT &acc) const {
    double yv[W], gv[W], pv[W], sv[W], rx[W];
    src.template ld<W>(S_Y, yqn, i, yv);
    src.template ld<W>(S_G, g, i, gv);
    src.template ld<W>(S_PX, px, i, pv);
    if (RX) {
      double a[W], b[W];
#pragma unroll
      for (int q = 0; q < W; q++) a[q] = b[q] = 0.0;
      if (zl) src.template ld<W>(S_ZL, zl, i, a);
      if (zu) src.template ld<W>(S_ZU, zu, i, b);
#pragma unroll
      for (int q = 0; q < W; q++) rx[q] = (a[q] - b[q]) - gv[q];
    }
    double ga[W];
#pragma unroll
    for (int q = 0; q < W; q++) {
      yv[q] += gv[q];
      ga[q] = gv[q];
    }
    for (int j = 0; j < ncon; j++) {
      double a[W];
      src.template ldc<W>(j, Acol.p[j], i, a);
#pragma unroll
      for (int q = 0; q < W; q++) {
        yv[q] = fma(-z.v[j], a[q], yv[q]);
        if (RX) rx[q] = fma(z.v[j], a[q], rx[q]);
        if (gaz) ga[q] = fma(-z.v[j], a[q], ga[q]);
      }
    }
    if (gaz) stv<W>(gaz, i, ga);
#pragma unroll
    for (int q = 0; q < W; q++) {
      yv[q] = fma(-coef[q], con.d[0], yv[q]);
      sv[q] = ax * pv[q];
      acc.s[0] = fma(yv[q], yv[q], acc.s[0]);
      acc.s[1] = fma(yv[q], sv[q], acc.s[1]);
      acc.s[2] = fma(sv[q], sv[q], acc.s[2]);
      if (RX) acc.x[0] = fmax(acc.x[0], fabs(fma(coef[q], con.d[0], rx[q])));
    }
    stv<W>(yqn, i, yv);
    stv<W>(sqn, i, sv);
  }
};
typedef Update2FT<0> Update2F;

// ============================================================== LinCombF
// out = beta * x + sum_j alpha_j V_j   (ParOptLBFGS::mult, QN.cpp:390-418, second
// pass; ParOptLSR1's Z_i = Y_i - b0 S_i, QN.cpp:730-735; damped-update vector).
// Traffic: reads (1 + ncols)N, writes N.
struct LinCombF : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *x;
  double beta;
  ColTable V;
  CoefTable alpha;
  int ncols;
  double *out;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(x);
    for (int j = 0; j < ncols; j++) p_(V.p[j]);
  }
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
    double o[W];
    if (x) {
      ldv<W>(x, i, o);
#pragma unroll
      for (int q = 0; q < W; q++) o[q] *= beta;
    } else {
#pragma unroll
      for (int q = 0; q < W; q++) o[q] = 0.0;
    }
    for (int j = 0; j < ncols; j++) {
      double c[W];
      ldv<W>(V.p[j], i, c);
#pragma unroll
      for (int q = 0; q < W; q++) o[q] = fma(alpha.v[j], c[q], o[q]);
    }
    stv<W>(out, i, o);
  }
};

// ============================================================== Pass1RF<MR>
// Pass1F fused with the reductions r_j = V_j . t1 (j < m <= MR) that the
// reference obtains with y.x->mdot(Ac) and step.x->mdot(Z) (IP.cpp:2142-2143,
// 2718): t1 never goes to memory.
// Traffic: reads (7 + m)N + 10W, writes N + W.   sums: 0..m-1 = [A|Z]^T t1
template <int MR>
struct Pass1RF : NoStreams {
  static constexpr int MINB = PCU_MINB_PASS1;
  static constexpr int NS = MR, NX = 0, NM = 0, NB = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // yw
  struct Elem {
    double d1, dinv;
  };
  DVars v, b;
  const double *lb, *ub, *Dinv, *Cw;
  double *d1, *d2;
  ColTable V;
  int m;
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(lb); p_(ub); p_(b.x); p_(Dinv);
    if (k.use_lower) p_(b.zl);
    if (k.use_upper) p_(b.zu);
    for (int j = 0; j < m; j++) p_(V.p[j]);
  }

  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1],
                                    AccT *) const {
    double x[W], l[W], u[W], bx[W], bzl[W], bzu[W], di[W], d[W];
    ldv<W>(v.x, i, x);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(b.x, i, bx);
    ldv<W>(Dinv, i, di);
#pragma unroll
    for (int q = 0; q < W; q++) bzl[q] = bzu[q] = 0.0;
    if (k.use_lower) ldv<W>(b.zl, i, bzl);
    if (k.use_upper) ldv<W>(b.zu, i, bzu);
#pragma unroll
    for (int q = 0; q < W; q++) {
      double t = bx[q];
      if (k.use_lower && l[q] > -k.mbv) t += bzl[q] / (x[q] - l[q]);
      if (k.use_upper && u[q] < k.mbv) t -= bzu[q] / (u[q] - x[q]);
      d[q] = t;
      e[q].d1 = t;
      e[q].dinv = di[q];
      part[q][0] = coef[q] * di[q] * t;
    }
    stv<W>(d1, i, d);
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1],
                                    Con &con, AccT &) const {
    const double sw = v.sw[ci], tw = v.tw[ci], zsw = v.zsw[ci], ztw = v.ztw[ci];
    const double dd = b.zw[ci] + (b.zsw[ci] + sw * b.sw[ci]) / zsw -
                      (b.ztw[ci] + tw * b.tw[ci]) / ztw;
    con.d[0] = Cw[ci] * (dd - sum[0]);
    d2[ci] = dd;
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AccT &acc) const {
    double t[W];
#pragma unroll
    for (int q = 0; q < W; q++) t[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
#pragma unroll
    for (int j = 0; j < MR; j++) {
      if (j < m) {
        double c[W];
        ldv<W>(V.p[j], i, c);
#pragma unroll
        for (int q = 0; q < W; q++) acc.s[j] = fma(t[q], c[q], acc.s[j]);
      }
    }
  }
};

// ============================================================== Pass2RF
// Pass2F that also emits the residual of the linearised KKT system at the step
// it has just produced (computeKKTRes + addKKTResStep, IP.cpp:1337-1583): the
// right-hand side of the next iterative-refinement solve (IP.cpp:4985-4991)
// costs one extra read (g) and three extra writes instead of a separate pass
// over (9 + c + q)N words.  The residual is written into the bundle `b` the
// right-hand side was read from (each entry is read before it is overwritten by
// the same thread).  beta_j = z_j + pz_j for the A columns and kap_k for the Z
// columns (B p = (b0 + sigma) p - Z kap), all for the accumulated step.
// Traffic: reads (10 + c + q)N + 20W, writes 6N + 10W (+3N + 5W reads when
// accumulating).
struct Pass2RF : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 1, NB2 = 2;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con2 Con;  // yw (this solve), zw + total pzw
  struct Elem {
    double d1, dinv, lin;
  };
  DVars v, b, y;
  const double *lb, *ub, *Dinv, *Cw, *d1, *d2, *g;
  ColTable V;
  CoefTable alpha, beta;
  int ncols;
  int accumulate;
  int from_vars;  // the right-hand side is computeKKTRes(vars, mu_rhs), recomputed
                  // here instead of being read from `b`
  double b0sig, mu, mu_rhs;
  IPConst k;
  // optional output: sum over the first nca columns (the constraint gradients) of
  // alpha_j V_j = A p_z of this solve; the update pass then forms -(g - A z+) from
  // g - A z (left by the previous update pass) without re-reading the nca columns
  double *apz = nullptr;
  int nca = 0;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(d1); p_(Dinv); p_(v.x); p_(lb); p_(ub); p_(g);
    if (k.use_lower) { p_(v.zl); if (!from_vars) p_(b.zl); }
    if (k.use_upper) { p_(v.zu); if (!from_vars) p_(b.zu); }
    for (int j = 0; j < ncols; j++) p_(V.p[j]);
    if (accumulate) {
      p_(y.x);
      if (k.use_lower) p_(y.zl);
      if (k.use_upper) p_(y.zu);
    }
  }

  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1],
                                    AccT *) const {
    double d[W], di[W], lin[W], qa[W];
    ldv<W>(d1, i, d);
    ldv<W>(Dinv, i, di);
#pragma unroll
    for (int q = 0; q < W; q++) lin[q] = qa[q] = 0.0;
    for (int j = 0; j < ncols; j++) {
      double c[W];
      ldv<W>(V.p[j], i, c);
#pragma unroll
      for (int q = 0; q < W; q++) {
        d[q] = fma(alpha.v[j], c[q], d[q]);
        lin[q] = fma(beta.v[j], c[q], lin[q]);
      }
      if (apz && j < nca) {
#pragma unroll
        for (int q = 0; q < W; q++) qa[q] = fma(alpha.v[j], c[q], qa[q]);
      }
    }
    if (apz) stv<W>(apz, i, qa);
#pragma unroll
    for (int q = 0; q < W; q++) {
      e[q].d1 = d[q];
      e[q].dinv = di[q];
      e[q].lin = lin[q];
      part[q][0] = coef[q] * di[q] * d[q];
    }
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1],
                                    Con &con, AccT &) const {
    const double yw = Cw[ci] * (d2[ci] - sum[0]);
    const double sw = v.sw[ci], tw = v.tw[ci], zsw = v.zsw[ci], ztw = v.ztw[ci];
    double bsw, btw, bzsw, bztw;
    if (from_vars) {  // IP.cpp:1361-1389
      const double zw = v.zw[ci];
      bsw = (zsw - gamma_sw(k, ci)) - zw;
      btw = (ztw - k.gamma) + zw;
      bzsw = mu_rhs - sw * zsw;
      bztw = mu_rhs - tw * ztw;
    } else {
      bsw = b.sw[ci];
      btw = b.tw[ci];
      bzsw = b.zsw[ci];
      bztw = b.ztw[ci];
    }
    const double pzsw = yw - bsw;
    const double pztw = -btw - yw;
    const double psw = (bzsw - sw * pzsw) / zsw;
    const double ptw = (bztw - tw * pztw) / ztw;
    double tzw = yw;
    if (accumulate) {
      tzw += y.zw[ci];
      y.zw[ci] = tzw;
      y.zsw[ci] += pzsw;
      y.ztw[ci] += pztw;
      y.sw[ci] += psw;
      y.tw[ci] += ptw;
    } else {
      y.zw[ci] = yw;
      y.zsw[ci] = pzsw;
      y.ztw[ci] = pztw;
      y.sw[ci] = psw;
      y.tw[ci] = ptw;
    }
    con.d[0] = yw;
    con.d[1] = v.zw[ci] + tzw;
  }
  template <int W>
  __device__ __forceinline__ void C2(long long i, const double (&coef)[W],
                                     const Elem (&e)[W], const Con &con, AccT &,
                                     double (&part2)[W][2]) const {
    double x[W], l[W], u[W], zl[W], zu[W], bzl[W], bzu[W], gv[W];
    double px[W], pzl[W], pzu[W], rx[W], rzl[W], rzu[W];
    ldv<W>(v.x, i, x);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = bzl[q] = bzu[q] = 0.0;
    if (k.use_lower) {
      ldv<W>(v.zl, i, zl);
      if (!from_vars) ldv<W>(b.zl, i, bzl);
    }
    if (k.use_upper) {
      ldv<W>(v.zu, i, zu);
      if (!from_vars) ldv<W>(b.zu, i, bzu);
    }
    if (from_vars) {  // rzl, rzu of computeKKTRes (IP.cpp:1417-1444)
#pragma unroll
      for (int q = 0; q < W; q++) {
        bzl[q] = -((x[q] - l[q]) * zl[q] - k.kappa * mu_rhs);
        bzu[q] = -((u[q] - x[q]) * zu[q] - k.kappa * mu_rhs);
      }
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      px[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
      pzl[q] = 0.0;
      pzu[q] = 0.0;
      if (k.use_lower && l[q] > -k.mbv)
        pzl[q] = (bzl[q] - zl[q] * px[q]) / (x[q] - l[q]);
      if (k.use_upper && u[q] < k.mbv)
        pzu[q] = (bzu[q] + zu[q] * px[q]) / (u[q] - x[q]);
    }
    if (accumulate) {
      double o[W];
      ldv<W>(y.x, i, o);
#pragma unroll
      for (int q = 0; q < W; q++) px[q] += o[q];
      if (k.use_lower) {
        ldv<W>(y.zl, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzl[q] += o[q];
      }
      if (k.use_upper) {
        ldv<W>(y.zu, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzu[q] += o[q];
      }
    }
    stv<W>(y.x, i, px);
    if (k.use_lower) stv<W>(y.zl, i, pzl);
    if (k.use_upper) stv<W>(y.zu, i, pzu);
    // residual of the linearised system at the (accumulated) step
#pragma unroll
    for (int q = 0; q < W; q++) {
      const double dl = x[q] - l[q], du = u[q] - x[q];
      double r = ((zl[q] - zu[q]) - gv[q]) + e[q].lin;
      r = fma(-b0sig, px[q], r) + (pzl[q] - pzu[q]);
      rx[q] = fma(coef[q], con.d[1], r);
      rzl[q] = 0.0;
      rzu[q] = 0.0;
      if (k.use_lower && l[q] > -k.mbv)
        rzl[q] = -(dl * zl[q] - k.kappa * mu) - (dl * pzl[q] + px[q] * zl[q]);
      if (k.use_upper && u[q] < k.mbv)
        rzu[q] = -(du * zu[q] - k.kappa * mu) - (du * pzu[q] - px[q] * zu[q]);
      part2[q][0] = coef[q] * x[q];
      part2[q][1] = coef[q] * px[q];
    }
    stv<W>(b.x, i, rx);
    if (k.use_lower) stv<W>(b.zl, i, rzl);
    if (k.use_upper) stv<W>(b.zu, i, rzu);
  }
  __device__ __forceinline__ void E(long long ci, const double (&sum2)[2],
                                    const Con &, AccT &) const {
    const double zw = v.zw[ci], sw = v.sw[ci], tw = v.tw[ci];
    const double zsw = v.zsw[ci], ztw = v.ztw[ci];
    const double pzw = y.zw[ci], psw = y.sw[ci], ptw = y.tw[ci];
    const double pzsw = y.zsw[ci], pztw = y.ztw[ci];
    const double gsw = gamma_sw(k, ci), gtw = k.gamma;
    b.zw[ci] = -(((wconst_at(k, ci) + sum2[0]) - sw) + tw) + ((psw - sum2[1]) - ptw);
    b.sw[ci] = ((zsw - gsw) - zw) + (pzsw - pzw);
    b.tw[ci] = ((ztw - gtw) + zw) + (pztw + pzw);
    b.zsw[ci] = (mu - sw * zsw) - (psw * zsw + sw * pzsw);
    b.ztw[ci] = (mu - tw * ztw) - (ptw * ztw + tw * pztw);
  }
};

// ============================================================== Pass2R1F<MR>
// Pass2RF fused with the first half of the NEXT (iterative-refinement) solve:
// the residual this pass produces is immediately turned into that solve's
// d1' / d2' (Pass1RF::A/B), its block solve t1' = D0^-1 (d1', d2')|x and the
// reductions [A|Z]^T t1' -- the columns of V are read once from HBM (the third
// round re-reads them through L1/L2 a few hundred cycles later).  Of the
// residual only the parts pass 2 of the next solve reads are stored (b.zl,
// b.zu, b.sw, b.tw, b.zsw, b.ztw); d1' goes to `d1out` (not in place: the
// generic path re-runs A).
// Traffic: reads (9 + c + q)N + 20W, writes 6N + 10W.   sums: [A|Z]^T t1'
struct Con3 {
  static constexpr int ND = 3;
  double d[3];
  // kept by the constraint's leader lane from B to E
  double zw, sw, tw, zsw, ztw, pzw, psw, ptw, pzsw, pztw;
  __device__ __forceinline__ void zero() { d[0] = d[1] = d[2] = 0.0; }
};
// WIDE = 1 (wide_tile_kernel, pcu_wide.cuh; MR = 0): the column sums of phase A arrive
// pre-added in the d1 slot and in the slot S_LIN of the stage, and phase F leaves t1'
// in the slot S_T for the kernel's column phase instead of walking the columns.
template <int MR, int WIDE = 0>
struct Pass2R1F : NoStreams {
  static constexpr int SRC = 1;
  static constexpr int MINB = PCU_MINB_PASS21;
  enum { S_D1, S_DINV, S_X, S_LB, S_UB, S_G, S_ZL, S_BZL, S_ZU, S_BZU, S_YX, S_YZL, S_YZU,
         S_LIN, S_T, S_V0 };
  static constexpr int NFIX = S_V0;  // fixed slots; the columns follow
  enum { W_CW, W_D2, W_SW, W_TW, W_ZSW, W_ZTW, W_ZW, W_BSW, W_BTW, W_BZSW, W_BZTW,
         W_YZW, W_YZSW, W_YZTW, W_YSW, W_YTW, NWSLOTS };
  static constexpr int NS = MR, NX = 0, NM = 0, NB = 1, NB2 = 3, NF = 1, FD = 2;
#if PCU_SMEMACC21
  // the MR running dot products live in shared memory (AccS): ~48 registers less
  static constexpr int SMEM = MR * PCU_TILE_THREADS * 8;
  typedef AccS<NS, NX, NM> AccT;
#else
  typedef Acc<NS, NX, NM> AccT;
#endif
  typedef Con3 Con;  // yw (this solve), zw + total pzw, yw' (next solve, first half)
  struct Elem {
    double d1, dinv, lin;
  };
  DVars v, b, y;
  const double *lb, *ub, *Dinv, *Cw, *d1, *g;
  double *d2, *d1out;
  ColTable V;
  CoefTable alpha, beta;
  // always -1 (the tables): the constant-bank operand form is kept because the
  // register allocation of this kernel depends on it (reading the tables directly
  // makes the register-fed Pass2R1F<16> spill)
  int cbank;
  int ncols;
  int accumulate;
  int from_vars;
  double b0sig, mu, mu_rhs;
  IPConst k;
  // optional output: sum over the first nca columns (the constraint gradients) of
  // alpha_j V_j = A p_z of this solve; the update pass then forms -(g - A z+) from
  // g - A z (left by the previous update pass) without re-reading the nca columns
  double *apz = nullptr;
  int nca = 0;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(d1); p_(Dinv); p_(v.x); p_(lb); p_(ub); p_(g);
    if (k.use_lower) { p_(v.zl); if (!from_vars) p_(b.zl); }
    if (k.use_upper) { p_(v.zu); if (!from_vars) p_(b.zu); }
    for (int j = 0; j < ncols; j++) p_(V.p[j]);
    if (accumulate) {
      p_(y.x);
      if (k.use_lower) p_(y.zl);
      if (k.use_upper) p_(y.zu);
    }
  }

  template <class P>
  __host__ __device__ __forceinline__ void tstreams(P &p_) const {
    p_.n(S_D1, d1); p_.n(S_DINV, Dinv); p_.n(S_X, v.x); p_.n(S_LB, lb); p_.n(S_UB, ub);
    p_.n(S_G, g);
    if (k.use_lower) { p_.n(S_ZL, v.zl); if (!from_vars) p_.n(S_BZL, b.zl); }
    if (k.use_upper) { p_.n(S_ZU, v.zu); if (!from_vars) p_.n(S_BZU, b.zu); }
    if (accumulate) {
      p_.n(S_YX, y.x);
      if (k.use_lower) p_.n(S_YZL, y.zl);
      if (k.use_upper) p_.n(S_YZU, y.zu);
    }
    for (int j = 0; j < ncols; j++) p_.n(S_V0 + j, V.p[j]);
    p_.w(W_CW, Cw); p_.w(W_D2, d2);
    p_.w(W_SW, v.sw); p_.w(W_TW, v.tw); p_.w(W_ZSW, v.zsw); p_.w(W_ZTW, v.ztw);
    p_.w(W_ZW, v.zw);
    if (!from_vars) {
      p_.w(W_BSW, b.sw); p_.w(W_BTW, b.tw); p_.w(W_BZSW, b.zsw); p_.w(W_BZTW, b.ztw);
    }
    if (accumulate) {
      p_.w(W_YZW, y.zw); p_.w(W_YZSW, y.zsw); p_.w(W_YZTW, y.ztw);
      p_.w(W_YSW, y.sw); p_.w(W_YTW, y.tw);
    }
  }

  template <int W, class S, class AT>
  __device__ __forceinline__ void A(const S &src, long long i, const double (&coef)[W],
                                    Elem (&e)[W], double (&part)[W][1],
                                    AT *) const {
    double d[W], di[W], lin[W], qa[W];
    src.template ld<W>(S_D1, d1, i, d);
    src.template ld<W>(S_DINV, Dinv, i, di);
#pragma unroll
    for (int q = 0; q < W; q++) lin[q] = qa[q] = 0.0;
    if constexpr (WIDE) src.template ld<W>(S_LIN, nullptr, i, lin);
    int j = 0;
    for (; j + 4 <= ncols; j += 4) {  // four columns per batch: loads first
      double c[4][W];
#pragma unroll
      for (int jj = 0; jj < 4; jj++) src.template ldc<W>(j + jj, V.p[j + jj], i, c[jj]);
      double al[4], be[4];
#pragma unroll
      for (int jj = 0; jj < 4; jj++) {
        al[jj] = pcu_coef(cbank, alpha, j + jj);
        be[jj] = pcu_coef(cbank >= 0 ? cbank + PCU_DENSE_MAXM : -1, beta, j + jj);
      }
#pragma unroll
      for (int jj = 0; jj < 4; jj++) {
#pragma unroll
        for (int q = 0; q < W; q++) {
          d[q] = fma(al[jj], c[jj][q], d[q]);
          lin[q] = fma(be[jj], c[jj][q], lin[q]);
        }
        if (apz && j + jj < nca) {
#pragma unroll
          for (int q = 0; q < W; q++) qa[q] = fma(al[jj], c[jj][q], qa[q]);
        }
      }
    }
    for (; j < ncols; j++) {
      double c[W];
      src.template ldc<W>(j, V.p[j], i, c);
      const double aj = pcu_coef(cbank, alpha, j);
      const double bj = pcu_coef(cbank >= 0 ? cbank + PCU_DENSE_MAXM : -1, beta, j);
#pragma unroll
      for (int q = 0; q < W; q++) {
        d[q] = fma(aj, c[q], d[q]);
        lin[q] = fma(bj, c[q], lin[q]);
      }
      if (apz && j < nca) {
#pragma unroll
        for (int q = 0; q < W; q++) qa[q] = fma(aj, c[q], qa[q]);
      }
    }
    if (apz) stv<W>(apz, i, qa);
#pragma unroll
    for (int q = 0; q < W; q++) {
      e[q].d1 = d[q];
      e[q].dinv = di[q];
      e[q].lin = lin[q];
      part[q][0] = coef[q] * di[q] * d[q];
    }
  }
  template <class S, class AT>
  __device__ __forceinline__ void B(const S &src, long long ci, const double (&sum)[1],
                                    Con &con, AT &) const {
    const double yw = src.ldw(W_CW, Cw, ci) * (src.ldw(W_D2, d2, ci) - sum[0]);
    const double sw = src.ldw(W_SW, v.sw, ci), tw = src.ldw(W_TW, v.tw, ci);
    const double zsw = src.ldw(W_ZSW, v.zsw, ci), ztw = src.ldw(W_ZTW, v.ztw, ci);
    const double zw = src.ldw(W_ZW, v.zw, ci);
    double bsw, btw, bzsw, bztw;
    if (from_vars) {  // IP.cpp:1361-1389
      bsw = (zsw - gamma_sw(k, ci)) - zw;
      btw = (ztw - k.gamma) + zw;
      bzsw = mu_rhs - sw * zsw;
      bztw = mu_rhs - tw * ztw;
    } else {
      bsw = src.ldw(W_BSW, b.sw, ci);
      btw = src.ldw(W_BTW, b.tw, ci);
      bzsw = src.ldw(W_BZSW, b.zsw, ci);
      bztw = src.ldw(W_BZTW, b.ztw, ci);
    }
    double pzsw = yw - bsw;
    double pztw = -btw - yw;
    double psw = pcu_div(bzsw - sw * pzsw, zsw);
    double ptw = pcu_div(bztw - tw * pztw, ztw);
    double tzw = yw;
    if (accumulate) {
      tzw += src.ldw(W_YZW, y.zw, ci);
      pzsw = src.ldw(W_YZSW, y.zsw, ci) + pzsw;
      pztw = src.ldw(W_YZTW, y.ztw, ci) + pztw;
      psw = src.ldw(W_YSW, y.sw, ci) + psw;
      ptw = src.ldw(W_YTW, y.tw, ci) + ptw;
    }
    y.zw[ci] = tzw;
    y.zsw[ci] = pzsw;
    y.ztw[ci] = pztw;
    y.sw[ci] = psw;
    y.tw[ci] = ptw;
    con.d[0] = yw;
    con.d[1] = zw + tzw;
    con.zw = zw; con.sw = sw; con.tw = tw; con.zsw = zsw; con.ztw = ztw;
    con.pzw = tzw; con.psw = psw; con.ptw = ptw; con.pzsw = pzsw; con.pztw = pztw;
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void C2(const S &src, long long i, const double (&coef)[W],
                                     Elem (&e)[W], const Con &con, AT &,
                                     double (&part2)[W][3]) const {
    double x[W], l[W], u[W], zl[W], zu[W], bzl[W], bzu[W], gv[W];
    double px[W], pzl[W], pzu[W], rzl[W], rzu[W], dn[W];
    src.template ld<W>(S_X, v.x, i, x);
    src.template ld<W>(S_LB, lb, i, l);
    src.template ld<W>(S_UB, ub, i, u);
    src.template ld<W>(S_G, g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = bzl[q] = bzu[q] = 0.0;
    if (k.use_lower) {
      src.template ld<W>(S_ZL, v.zl, i, zl);
      if (!from_vars) src.template ld<W>(S_BZL, b.zl, i, bzl);
    }
    if (k.use_upper) {
      src.template ld<W>(S_ZU, v.zu, i, zu);
      if (!from_vars) src.template ld<W>(S_BZU, b.zu, i, bzu);
    }
    if (from_vars) {  // rzl, rzu of computeKKTRes (IP.cpp:1417-1444)
#pragma unroll
      for (int q = 0; q < W; q++) {
        bzl[q] = -((x[q] - l[q]) * zl[q] - k.kappa * mu_rhs);
        bzu[q] = -((u[q] - x[q]) * zu[q] - k.kappa * mu_rhs);
      }
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      px[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
      pzl[q] = 0.0;
      pzu[q] = 0.0;
      if (k.use_lower && l[q] > -k.mbv)
        pzl[q] = pcu_div(bzl[q] - zl[q] * px[q], x[q] - l[q]);
      if (k.use_upper && u[q] < k.mbv)
        pzu[q] = pcu_div(bzu[q] + zu[q] * px[q], u[q] - x[q]);
    }
    if (accumulate) {
      double o[W];
      src.template ld<W>(S_YX, y.x, i, o);
#pragma unroll
      for (int q = 0; q < W; q++) px[q] += o[q];
      if (k.use_lower) {
        src.template ld<W>(S_YZL, y.zl, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzl[q] += o[q];
      }
      if (k.use_upper) {
        src.template ld<W>(S_YZU, y.zu, i, o);
#pragma unroll
        for (int q = 0; q < W; q++) pzu[q] += o[q];
      }
    }
    stv<W>(y.x, i, px);
    if (k.use_lower) stv<W>(y.zl, i, pzl);
    if (k.use_upper) stv<W>(y.zu, i, pzu);
    // residual of the linearised system at the (accumulated) step, and the
    // first half of the diagonal solve on it (IP.cpp:2091-2107)
#pragma unroll
    for (int q = 0; q < W; q++) {
      const double dl = x[q] - l[q], du = u[q] - x[q];
      double r = ((zl[q] - zu[q]) - gv[q]) + e[q].lin;
      r = fma(-b0sig, px[q], r) + (pzl[q] - pzu[q]);
      double t = fma(coef[q], con.d[1], r);  // rx
      rzl[q] = 0.0;
      rzu[q] = 0.0;
      if (k.use_lower && l[q] > -k.mbv) {
        rzl[q] = -(dl * zl[q] - k.kappa * mu) - (dl * pzl[q] + px[q] * zl[q]);
        t += pcu_div(rzl[q], dl);
      }
      if (k.use_upper && u[q] < k.mbv) {
        rzu[q] = -(du * zu[q] - k.kappa * mu) - (du * pzu[q] - px[q] * zu[q]);
        t -= pcu_div(rzu[q], du);
      }
      dn[q] = t;
      e[q].d1 = t;
      part2[q][0] = coef[q] * x[q];
      part2[q][1] = coef[q] * px[q];
      part2[q][2] = coef[q] * e[q].dinv * t;
    }
    stv<W>(d1out, i, dn);
    if (k.use_lower) stv<W>(b.zl, i, rzl);
    if (k.use_upper) stv<W>(b.zu, i, rzu);
  }
  template <class S, class AT>
  __device__ __forceinline__ void E(const S &src, long long ci, const double (&sum2)[3],
                                    Con &con, AT &) const {
    const double zw = con.zw, sw = con.sw, tw = con.tw;
    const double zsw = con.zsw, ztw = con.ztw;
    const double pzw = con.pzw, psw = con.psw, ptw = con.ptw;
    const double pzsw = con.pzsw, pztw = con.pztw;
    const double gsw = gamma_sw(k, ci), gtw = k.gamma;
    const double bzw = -(((wconst_at(k, ci) + sum2[0]) - sw) + tw) + ((psw - sum2[1]) - ptw);
    const double bsw = ((zsw - gsw) - zw) + (pzsw - pzw);
    const double btw = ((ztw - gtw) + zw) + (pztw + pzw);
    const double bzsw = (mu - sw * zsw) - (psw * zsw + sw * pzsw);
    const double bztw = (mu - tw * ztw) - (ptw * ztw + tw * pztw);
    b.sw[ci] = bsw;
    b.tw[ci] = btw;
    b.zsw[ci] = bzsw;
    b.ztw[ci] = bztw;
    const double dd = bzw + pcu_div(bzsw + sw * bsw, zsw) - pcu_div(bztw + tw * btw, ztw);
    d2[ci] = dd;
    con.d[2] = src.ldw(W_CW, Cw, ci) * (dd - sum2[2]);
  }
  template <int W, class S, class AT>
  __device__ __forceinline__ void F(const S &src, long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AT &acc) const {
    double t[W];
#pragma unroll
    for (int q = 0; q < W; q++) t[q] = e[q].dinv * fma(coef[q], con.d[2], e[q].d1);
    if constexpr (WIDE) src.template st<W>(S_T, i, t);
    // eight columns at a time: the loads of a batch are issued before the
    // dependent multiply-adds (this loop held 18 % of the kernel's stall samples)
#pragma unroll
    for (int j0 = 0; j0 < (WIDE ? 0 : MR); j0 += 8) {
      if (j0 < ncols) {
        double c[8][W];
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
#pragma unroll
          for (int q = 0; q < W; q++) c[jj][q] = 0.0;
          if (j0 + jj < ncols) src.template ldc<W>(j0 + jj, V.p[j0 + jj], i, c[jj]);
        }
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
#pragma unroll
          for (int q = 0; q < W; q++) acc.s[j0 + jj] = fma(t[q], c[jj][q], acc.s[j0 + jj]);
        }
      }
    }
  }
  template <class S, class AT>
  __device__ __forceinline__ void FG(const S &, long long i, double coef, const Con &con,
                                     AT &acc) const {
    const double t = Dinv[i] * fma(coef, con.d[2], d1out[i]);
#pragma unroll
    for (int j = 0; j < MR; j++) {
      if (j < ncols) acc.s[j] = fma(t, V.p[j][i], acc.s[j]);
    }
  }
};

// ============================================================== Pass1VF<MR>
// Pass1RF whose right-hand side is the KKT residual itself (computeKKTRes,
// IP.cpp:1337-1446, at barrier mu), recomputed from the variables: the first
// solve of an iteration never reads (and ResF never writes) the residual
// vectors.  Traffic: reads (8 + c + m)N + 6W, writes N + W.
template <int MR>
struct Pass1VF : NoStreams {
  static constexpr int MINB = PCU_MINB_PASS1;
  static constexpr int NS = MR, NX = 0, NM = 0, NB = 2, HASP = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con2 Con;  // yw, zw
  struct Elem {
    double d1, dinv;
  };
  DVars v;
  const double *lb, *ub, *g, *Dinv, *Cw;
  double *d1, *d2;
  ColTable V;   // [A | Z]; the first ncon columns are the constraint gradients
  CoefTable z;  // dense multipliers
  int m, ncon;
  double mu;
  IPConst k;

  template <class P>
  __device__ __forceinline__ void streams(P &p_) const {
    p_(v.x); p_(lb); p_(ub); p_(g); p_(Dinv);
    if (k.use_lower) p_(v.zl);
    if (k.use_upper) p_(v.zu);
    for (int j = 0; j < m; j++) p_(V.p[j]);
  }
  __device__ __forceinline__ void P(long long ci, Con &con) const {
    con.d[1] = v.zw[ci];
  }
  template <int W>
  __device__ __forceinline__ void AP(long long i, const double (&coef)[W],
                                     Elem (&e)[W], double (&part)[W][2], AccT *,
                                     const Con &con) const {
    double x[W], l[W], u[W], gv[W], zl[W], zu[W], di[W], d[W];
    ldv<W>(v.x, i, x);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(g, i, gv);
    ldv<W>(Dinv, i, di);
#pragma unroll
    for (int q = 0; q < W; q++) zl[q] = zu[q] = 0.0;
    if (k.use_lower) ldv<W>(v.zl, i, zl);
    if (k.use_upper) ldv<W>(v.zu, i, zu);
#pragma unroll
    for (int q = 0; q < W; q++) d[q] = (zl[q] - zu[q]) - gv[q];
    for (int j = 0; j < ncon; j++) {
      double a[W];
      ldv<W>(V.p[j], i, a);
#pragma unroll
      for (int q = 0; q < W; q++) d[q] = fma(z.v[j], a[q], d[q]);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      const double dl = x[q] - l[q], du = u[q] - x[q];
      double t = fma(coef[q], con.d[1], d[q]);  // rx
      if (k.use_lower && l[q] > -k.mbv) t += -(dl * zl[q] - k.kappa * mu) / dl;
      if (k.use_upper && u[q] < k.mbv) t -= -(du * zu[q] - k.kappa * mu) / du;
      d[q] = t;
      e[q].d1 = t;
      e[q].dinv = di[q];
      part[q][0] = coef[q] * di[q] * t;
      part[q][1] = coef[q] * x[q];
    }
    stv<W>(d1, i, d);
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[2],
                                    Con &con, AccT &) const {
    const double zw = v.zw[ci], sw = v.sw[ci], tw = v.tw[ci];
    const double zsw = v.zsw[ci], ztw = v.ztw[ci];
    const double bzw = -(((wconst_at(k, ci) + sum[1]) - sw) + tw);
    const double bsw = (zsw - gamma_sw(k, ci)) - zw;
    const double btw = (ztw - k.gamma) + zw;
    const double bzsw = mu - sw * zsw;
    const double bztw = mu - tw * ztw;
    const double dd = bzw + (bzsw + sw * bsw) / zsw - (bztw + tw * btw) / ztw;
    con.d[0] = Cw[ci] * (dd - sum[0]);
    con.d[1] = zw;
    d2[ci] = dd;
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&coef)[W],
                                    const Elem (&e)[W], const Con &con,
                                    AccT &acc) const {
    double t[W];
#pragma unroll
    for (int q = 0; q < W; q++) t[q] = e[q].dinv * fma(coef[q], con.d[0], e[q].d1);
#pragma unroll
    for (int j = 0; j < MR; j++) {
      if (j < m) {
        double c[W];
        ldv<W>(V.p[j], i, c);
#pragma unroll
        for (int q = 0; q < W; q++) acc.s[j] = fma(t[q], c[q], acc.s[j]);
      }
    }
  }
};
