// pcu_dense.cuh -- the small dense algebra of the KKT solve (the c x c matrix G,
// the q x q matrix Ce, the Sherman-Morrison-Woodbury coefficients) as ONE piece of
// host/device code, so that the default iteration's solve
//     Gram pass -> [pcu_dense_solve] -> Pass2SVF (the step + its statistics)
// runs either on the device without a host round trip (pcu_dense.cu: single-CTA kernel
// on a flat work buffer staged in shared memory) or, with the same statements, on the
// host (pcu_dense_host).  The one iterative-refinement step of that solve is done here,
// in the column space of V = [A|Z] (pcu_dense_solve).  Every other route of the host
// (pcu_ip::setUpKKTSystem, computeKKTStep, the GMRES preconditioner, the starting points,
// the quasi-Newton M) calls the same functions, on any width up to PCU_MAX_COLS, and
// keeps its factors in the same flat buffer.  Reference: setUpKKTDiagSystem's
// G (IP.cpp:1932-1969, dgetrf), setUpKKTSystem's Ce (IP.cpp:2646-2664, dgetrf), the
// dense part of solveKKTDiagSystem (IP.cpp:2150-2170, 2288-2306) and of computeKKTStep
// (IP.cpp:2716-2735), computeKKTRes / addKKTResStep's dense residual
// (IP.cpp:1401-1407, 1535-1541), ParOptLBFGS::mult's compact solve (QN.cpp:398-412),
// the refinement loop (IP.cpp:4985-4991).
//
// The device replaces the divisions on its critical path by reciprocals (<= 1 ulp
// each), so the device and host runs agree to round-off (tests/test_gpu_gram_paths.py
// holds the two histories to 1e-12).  The host divides, as LAPACK does.
#pragma once

#include <cuda_runtime.h>

#define PCU_DENSE_MAXM 32  // chain mode: ncon + quasi-Newton width <= 32 (ld <= 40)
#define PCU_HD __host__ __device__ __forceinline__
// The dense kernel runs ONCE per launch in a single warp: its cost is instruction
// fetch (cold instruction cache), not arithmetic -- 10.5k SASS instructions of fully
// inlined / unrolled code took 200k cycles per launch.  The building blocks are
// therefore real functions (one copy each, warm after their first call) with rolled
// loops, and the fp64 divisions are the short reciprocal sequence below.
#define PCU_HDN static __host__ __device__ __noinline__

// Offsets (in doubles) into the flat work buffer.  [0, S) is written by the host
// before the chain (inputs), [S, total) is produced on the device and read back.
// m <= PCU_DENSE_MAXM on the device; the host routes take up to PCU_MAX_COLS columns.
struct DenseOff {
  int c, q, ld, m;
  int mu, vz, vs, vt, vzs, vzt, cc, gs, gt;  // inputs: barrier, dense variables, c(x), penalties
  int M, d0, Mf, mpiv;                       // quasi-Newton compact matrix, its LU and pivots
  int S;                                     // symmetrised Gram matrix (ld x ld)
  int Graw, Gfac, gpiv, Ceraw, Cefac, cpiv;
  int ginv, ceinv, minv;                     // reciprocal diagonals of the three LU factors
  int bz, bs, bt, bzs, bzt;                  // dense residual (right-hand side)
  int yz, ys, yt, yzs, yzt;                  // dense step (accumulated)
  int r, vtp;                                // [A|Z]^T t1 of the current solve; [A|Z]^T step
  int coef, alpha2;                          // alpha of the first solve, then of the whole step
                                             // (the pass's table); alpha of the refinement
  int total;
};

static inline DenseOff pcu_dense_offsets(int c, int q, int ld) {
  DenseOff o;
  o.c = c;
  o.q = q;
  o.ld = ld;
  o.m = c + q;
  int p = 0;
  auto take = [&p](int n) {
    const int at = p;
    p += n;
    return at;
  };
  o.mu = take(2);
  o.vz = take(c); o.vs = take(c); o.vt = take(c); o.vzs = take(c); o.vzt = take(c);
  o.cc = take(c); o.gs = take(c); o.gt = take(c);
  o.M = take(q * q); o.d0 = take(q); o.Mf = take(q * q); o.mpiv = take(q);
  p = (p + 1) & ~1;
  o.S = take(ld * ld);
  o.Graw = take(c * c); o.Gfac = take(c * c); o.gpiv = take(c);
  o.Ceraw = take(q * q); o.Cefac = take(q * q); o.cpiv = take(q);
  o.ginv = take(c); o.ceinv = take(q); o.minv = take(q);
  o.bz = take(c); o.bs = take(c); o.bt = take(c); o.bzs = take(c); o.bzt = take(c);
  o.yz = take(c); o.ys = take(c); o.yt = take(c); o.yzs = take(c); o.yzt = take(c);
  o.r = take(o.m); o.vtp = take(o.m);
  p = (p + 1) & ~1;
  const int ncoef = o.m > PCU_DENSE_MAXM ? o.m : PCU_DENSE_MAXM;  // >= the constant bank
  o.coef = take(ncoef);
  o.alpha2 = take(ncoef);
  o.total = (p + 1) & ~1;
  return o;
}

// ---------------------------------------------------------------- lane model
// The phases below are written once for the host (one "lane", no barrier) and for the
// device, where ONE WARP runs them on the shared-memory copy of the buffer: loops whose
// iterations are independent are dealt over the lanes (PCU_PFOR) and separated by
// __syncwarp(); every element still sees the host's sequence of operations.
#ifdef __CUDA_ARCH__
#define PCU_LANE ((int)(threadIdx.x & 31))
#define PCU_NLANE 32
#define PCU_SYNC() __syncwarp()
#else
#define PCU_LANE 0
#define PCU_NLANE 1
#define PCU_SYNC() ((void)0)
#endif
#define PCU_PFOR(i, lo, hi) \
  _Pragma("unroll 1") for (int i = (lo) + PCU_LANE; i < (hi); i += PCU_NLANE)
// optional device-side profile of the phases (PCU_DENSE_TICKS): clock64 at checkpoints
#ifdef __CUDA_ARCH__
#define PCU_TICK(t, k) do { if ((t) && PCU_LANE == 0) (t)[k] = clock64(); } while (0)
#else
#define PCU_TICK(t, k) ((void)0)
#endif
// doubles of scratch the phases need next to the buffer
#define PCU_DENSE_SCRATCH(c, q) ((c) * (q) + 2 * ((c) + (q)) + 5 * (c) + (q) + 8)

// 1 / x.  On the device the divisions of the factorisations and triangular solves sit
// on the critical path of a single warp (an IEEE fp64 division is a ~25-instruction
// dependent sequence): the hardware seed + two Newton steps (<= 1 ulp) replaces it,
// and the triangular solves multiply by reciprocal diagonals computed once per factor.
PCU_HDN double pcu_dense_rcp(double x) {
#ifdef __CUDA_ARCH__
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
#else
  return 1.0 / x;
#endif
}

PCU_HDN double pcu_dense_div(double a, double b) {
#ifdef __CUDA_ARCH__
  const double r = pcu_dense_rcp(b);
  const double q = a * r;
  return fma(fma(-b, q, a), r, q);  // one residual correction: <= 1 ulp
#else
  return a / b;
#endif
}

// LAPACK dgetrf / dgetrs restated (partial pivoting, first largest entry, column-major;
// n <= 32 on the device, any n on the host); pivots are kept as doubles inside the flat
// buffer, invd receives the reciprocal diagonal.  The solves read invd on the device only
// (the host divides by the diagonal and may pass NULL).
PCU_HDN int pcu_dense_lu_factor(int n, double *A, double *piv, double *invd) {
  int info = 0;
#pragma unroll 1
  for (int k = 0; k < n; k++) {
    int p = k;
#ifdef __CUDA_ARCH__
    {
      const int i = k + PCU_LANE;
      double v = i < n ? fabs(A[i + n * k]) : -1.0;
      int idx = i < n ? i : n;
#pragma unroll 1
      for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        if (v2 > v || (v2 == v && i2 < idx)) {
          v = v2;
          idx = i2;
        }
      }
      p = idx;
    }
#else
    double best = fabs(A[k + n * k]);
#pragma unroll 1
    for (int i = k + 1; i < n; i++) {
      const double v = fabs(A[i + n * k]);
      if (v > best) {
        best = v;
        p = i;
      }
    }
#endif
    if (PCU_LANE == 0) piv[k] = (double)p;
    const double pivot = A[p + n * k];
    PCU_SYNC();  // every lane has read the pivot before the rows are exchanged
    if (pivot == 0.0) {
      if (!info) info = k + 1;
      if (PCU_LANE == 0) invd[k] = 0.0;
      continue;
    }
    if (p != k) {
      PCU_PFOR(j, 0, n) {
        const double t = A[k + n * j];
        A[k + n * j] = A[p + n * j];
        A[p + n * j] = t;
      }
      PCU_SYNC();
    }
    const double inv = pcu_dense_rcp(pivot);
    if (PCU_LANE == 0) invd[k] = inv;
    PCU_PFOR(i, k + 1, n) A[i + n * k] *= inv;
    PCU_SYNC();
    // trailing update: a lane owns row i (n <= 32), its multiplier stays in a register;
    // the host runs down the columns (the same operation on every element)
#ifdef __CUDA_ARCH__
    PCU_PFOR(i, k + 1, n) {
      const double lik = A[i + n * k];
#pragma unroll 1
      for (int j = k + 1; j < n; j++) {
        const double akj = A[k + n * j];
        if (akj != 0.0) A[i + n * j] -= lik * akj;
      }
    }
#else
    for (int j = k + 1; j < n; j++) {
      const double akj = A[k + n * j];
      if (akj != 0.0)
        for (int i = k + 1; i < n; i++) A[i + n * j] -= A[i + n * k] * akj;
    }
#endif
    PCU_SYNC();
  }
  return info;
}

PCU_HDN void pcu_dense_lu_solve(int n, const double *LU, const double *piv, const double *invd,
                               double *b) {
  if (PCU_LANE == 0) {
#pragma unroll 1
    for (int k = 0; k < n; k++) {
      const int p = (int)piv[k];
      if (p != k) {
        const double t = b[k];
        b[k] = b[p];
        b[p] = t;
      }
    }
  }
  PCU_SYNC();
#pragma unroll 1
  for (int k = 0; k < n; k++) {
    const double bk = b[k];
    if (bk != 0.0) {
      PCU_PFOR(i, k + 1, n) b[i] -= LU[i + n * k] * bk;
    }
    PCU_SYNC();
  }
#pragma unroll 1
  for (int k = n - 1; k >= 0; k--) {
#ifdef __CUDA_ARCH__
    if (PCU_LANE == 0) b[k] *= invd[k];
#else
    b[k] /= LU[k + n * k];
#endif
    PCU_SYNC();
    const double bk = b[k];
    PCU_PFOR(i, 0, k) b[i] -= LU[i + n * k] * bk;
    PCU_SYNC();
  }
}

// The same solve run by ONE lane on its own right-hand side (several independent
// solves side by side).
PCU_HDN void pcu_dense_lu_solve_lane(int n, const double *LU, const double *piv,
                                    const double *invd, double *b) {
#pragma unroll 1
  for (int k = 0; k < n; k++) {
    const int p = (int)piv[k];
    if (p != k) {
      const double t = b[k];
      b[k] = b[p];
      b[p] = t;
    }
  }
#pragma unroll 1
  for (int k = 0; k < n; k++) {
    const double bk = b[k];
    if (bk != 0.0) {
#pragma unroll 1
      for (int i = k + 1; i < n; i++) b[i] -= LU[i + n * k] * bk;
    }
  }
#pragma unroll 1
  for (int k = n - 1; k >= 0; k--) {
#ifdef __CUDA_ARCH__
    b[k] *= invd[k];
#else
    b[k] /= LU[k + n * k];
#endif
    const double bk = b[k];
#pragma unroll 1
    for (int i = 0; i < k; i++) b[i] -= LU[i + n * k] * bk;
  }
}

// Dense residual of computeKKTRes (with_step = 0) / addKKTResStep (with_step = 1:
// the step is w[yz..], [A|Z]^T px is w[vtp]).
PCU_HDN void pcu_dense_residual(double *w, const DenseOff &o, int with_step) {
  const double mu = w[o.mu];
  PCU_PFOR(i, 0, o.c) {
    const double z = w[o.vz + i], s = w[o.vs + i], t = w[o.vt + i];
    const double zs = w[o.vzs + i], zt = w[o.vzt + i];
    double rz = -(w[o.cc + i] - s + t);
    double rs = -(w[o.gs + i] - zs + z);
    double rt = -(w[o.gt + i] - zt - z);
    double rzs = -(s * zs - mu);
    double rzt = -(t * zt - mu);
    if (with_step) {
      const double pz = w[o.yz + i], ps = w[o.ys + i], pt = w[o.yt + i];
      const double pzs = w[o.yzs + i], pzt = w[o.yzt + i];
      rz -= (w[o.vtp + i] - ps + pt);
      rs += (pzs - pz);
      rt += (pzt + pz);
      rzs -= (ps * zs + s * pzs);
      rzt -= (pt * zt + t * pzt);
    }
    w[o.bz + i] = rz;
    w[o.bs + i] = rs;
    w[o.bt + i] = rt;
    w[o.bzs + i] = rzs;
    w[o.bzt + i] = rzt;
  }
  PCU_SYNC();
}

// G = C0 + S_AA, Ce = S_ZZ - S_ZA G^-1 S_AZ - M / (d d^T), both LU-factored
// (IP.cpp:1932-1969, 2646-2664).  scratch: >= c * q doubles.
PCU_HDN void pcu_dense_setup(double *w, const DenseOff &o, double *scratch) {
  const int c = o.c, q = o.q, ld = o.ld, m = o.m;
  double *S = w + o.S;
  PCU_PFOR(i, 0, m) {  // symmetrise from the lower triangle (a lane owns row i)
#pragma unroll 1
    for (int j = 0; j < i; j++) S[j + ld * i] = S[i + ld * j];
  }
  PCU_SYNC();
  double *Graw = w + o.Graw, *Gfac = w + o.Gfac;
  PCU_PFOR(i, 0, c) {
#pragma unroll 1
    for (int j = 0; j < c; j++) {
      double g = S[i + ld * j];
      if (i == j)
        g += pcu_dense_div(w[o.vs + i], w[o.vzs + i]) + pcu_dense_div(w[o.vt + i], w[o.vzt + i]);
      Graw[i + c * j] = g;
      Gfac[i + c * j] = g;
    }
  }
  PCU_SYNC();
  if (c > 0) pcu_dense_lu_factor(c, Gfac, w + o.gpiv, w + o.ginv);
  if (q > 0) {
    double *Ceraw = w + o.Ceraw, *Cefac = w + o.Cefac;
    // column i of G^-1 S_AZ, one lane per column
    PCU_PFOR(i, 0, q) {
      double *col = scratch + c * i;
#pragma unroll 1
      for (int j = 0; j < c; j++) col[j] = S[j + ld * (c + i)];
      if (c > 0) pcu_dense_lu_solve_lane(c, Gfac, w + o.gpiv, w + o.ginv, col);
    }
    PCU_SYNC();
    const double *M = w + o.M, *d0 = w + o.d0;
    PCU_PFOR(k, 0, q) {  // a lane owns row k
#pragma unroll 1
      for (int i = 0; i < q; i++) {
        const double *col = scratch + c * i;
        double v = S[(c + k) + ld * (c + i)];
#pragma unroll 1
        for (int j = 0; j < c; j++) v -= S[(c + k) + ld * j] * col[j];
        v -= pcu_dense_div(M[k + q * i], d0[k] * d0[i]);
        Ceraw[k + q * i] = v;
        Cefac[k + q * i] = v;
      }
    }
    PCU_SYNC();
    pcu_dense_lu_factor(q, Cefac, w + o.cpiv, w + o.ceinv);
  }
}

// Dense half of computeKKTStep on the right-hand side w[bz..] with the reductions
// w[r]: SMW coefficients into `alpha` (m values), the dense step into w[yz..]
// (added when accumulate), w[vtp] = (accumulate ? vtp : 0) + r + S alpha.
// scratch: >= 2 m + 5 c doubles.
PCU_HDN void pcu_dense_step(double *w, const DenseOff &o, int accumulate, double *alpha,
                           double *scratch) {
  const int c = o.c, q = o.q, ld = o.ld, m = o.m;
  const double *S = w + o.S, *r = w + o.r;
  double *yz1 = scratch, *pz = yz1 + c, *ps = pz + c, *pt = ps + c, *pzs = pt + c;
  double *pzt = pzs + c, *ww = pzt + c, *yz2 = ww + q;
  PCU_PFOR(i, 0, c) {
    const double s = w[o.vs + i], t = w[o.vt + i], zs = w[o.vzs + i], zt = w[o.vzt + i];
    yz1[i] = (w[o.bz + i] + pcu_dense_div(w[o.bzs + i] + s * w[o.bs + i], zs) -
              pcu_dense_div(w[o.bzt + i] + t * w[o.bt + i], zt) - r[i]);
  }
  PCU_SYNC();
  if (c > 0) pcu_dense_lu_solve(c, w + o.Gfac, w + o.gpiv, w + o.ginv, yz1);
  PCU_PFOR(i, 0, c) {
    const double s = w[o.vs + i], t = w[o.vt + i], zs = w[o.vzs + i], zt = w[o.vzt + i];
    pz[i] = yz1[i];
    pzs[i] = yz1[i] - w[o.bs + i];
    pzt[i] = -w[o.bt + i] - yz1[i];
    ps[i] = pcu_dense_div(w[o.bzs + i] - s * pzs[i], zs);
    pt[i] = pcu_dense_div(w[o.bzt + i] - t * pzt[i], zt);
    alpha[i] = yz1[i];
  }
  PCU_SYNC();
  if (q > 0) {
    PCU_PFOR(kq, 0, q) {  // Z^T yx = r_Z + S_ZA yz1
      double v = r[c + kq];
#pragma unroll 1
      for (int j = 0; j < c; j++) v += S[(c + kq) + ld * j] * yz1[j];
      ww[kq] = v;
    }
    PCU_SYNC();
    pcu_dense_lu_solve(q, w + o.Cefac, w + o.cpiv, w + o.ceinv, ww);
    PCU_PFOR(j, 0, c) {  // second solve: A^T P Z w = S_AZ w
      double v = 0.0;
#pragma unroll 1
      for (int kq = 0; kq < q; kq++) v += S[j + ld * (c + kq)] * ww[kq];
      yz2[j] = -v;
    }
    PCU_SYNC();
    if (c > 0) pcu_dense_lu_solve(c, w + o.Gfac, w + o.gpiv, w + o.ginv, yz2);
    PCU_PFOR(i, 0, c) {
      const double s = w[o.vs + i], t = w[o.vt + i], zs = w[o.vzs + i], zt = w[o.vzt + i];
      const double yzs2 = yz2[i], yzt2 = -yz2[i];
      const double ys2 = pcu_dense_div(-(s * yzs2), zs);
      const double yt2 = pcu_dense_div(-(t * yzt2), zt);
      pz[i] -= yz2[i];
      pzs[i] -= yzs2;
      pzt[i] -= yzt2;
      ps[i] -= ys2;
      pt[i] -= yt2;
      alpha[i] = pz[i];
    }
    PCU_PFOR(kq, 0, q) alpha[c + kq] = -ww[kq];
    PCU_SYNC();
  }
  PCU_PFOR(i, 0, c) {
    if (accumulate) {
      w[o.yz + i] += pz[i];
      w[o.ys + i] += ps[i];
      w[o.yt + i] += pt[i];
      w[o.yzs + i] += pzs[i];
      w[o.yzt + i] += pzt[i];
    } else {
      w[o.yz + i] = pz[i];
      w[o.ys + i] = ps[i];
      w[o.yt + i] = pt[i];
      w[o.yzs + i] = pzs[i];
      w[o.yzt + i] = pzt[i];
    }
  }
  PCU_PFOR(i, 0, m) {  // [A|Z]^T D0^-1 (d1 + V alpha) = r + S alpha
    double vv = r[i];
#pragma unroll 1
    for (int j = 0; j < m; j++) vv += S[i + ld * j] * alpha[j];
    w[o.vtp + i] = accumulate ? w[o.vtp + i] + vv : vv;
  }
  PCU_SYNC();
}

// The KKT solve of the default iteration (one refinement step) between the Gram pass and
// the one pass that applies it.  w[S] holds the Gram result (ld x ld, lower triangle,
// row m = [A|Z]^T t1 of the first solve, t1 = D0^-1 d1).  scratch: >= max(c q, 2 m + 5 c).
//
// The first solve is p1 = D0^-1 (d1 + V alpha1), V = [A|Z].  The x row of its
// residual r - K p1 is (Pass2R1F's rx with lin = V beta, beta = (z + pz, kap))
//     t = A (pz - alpha1_A) + Z (kap - alpha1_Z) = V delta,
//     delta_A = 0 exactly (alpha1_A is pz),  delta_Z = kap - alpha1_Z,
// and the bound and weighting rows of that residual vanish given px.  So the
// refinement solve's reductions are r' = V^T D0^-1 t = S delta, its dense rows are the
// dense residual at p1, and the refined step is
//     p = p1 + D0^-1 (t + V alpha2) = D0^-1 (d1 + V (alpha1 + delta + alpha2)):
// one pass with the table (alpha1_A + alpha2_A, kap + alpha2_Z) left in w[coef].  What
// this drops against refining the N-sized residual elementwise is the rounding of the
// elementwise operations (relative eps per element); the correction the refinement is
// for -- the error of the solves with G and Ce -- lives in this column space and is kept.
PCU_HD void pcu_dense_solve(double *w, const DenseOff &o, double *scratch,
                            long long *tick = nullptr) {
  const int c = o.c, q = o.q, ld = o.ld, m = o.m;
  PCU_PFOR(j, 0, m) w[o.r + j] = w[o.S + m + ld * j];
  PCU_SYNC();
  pcu_dense_setup(w, o, scratch);
  PCU_TICK(tick, 2);
  pcu_dense_residual(w, o, 0);
  double *alpha = w + o.coef, *alpha2 = w + o.alpha2;
  pcu_dense_step(w, o, 0, alpha, scratch);
  PCU_TICK(tick, 3);
  // kap = d0 M^-1 d0 (Z^T p1), the compact quasi-Newton solve (IP.cpp:1474-1476):
  // alpha_Z takes kap, alpha2_Z holds delta_Z until the refinement step overwrites it
  if (q > 0) {
    double *kap = alpha2 + c;
    PCU_PFOR(i, 0, q) {
      kap[i] = w[o.vtp + c + i] * w[o.d0 + i];
      w[o.minv + i] = pcu_dense_rcp(w[o.Mf + i * (q + 1)]);
    }
    PCU_SYNC();
    pcu_dense_lu_solve(q, w + o.Mf, w + o.mpiv, w + o.minv, kap);
    PCU_PFOR(i, 0, q) {
      const double kz = kap[i] * w[o.d0 + i];
      kap[i] = kz - alpha[c + i];
      alpha[c + i] = kz;
    }
  }
  PCU_SYNC();
  pcu_dense_residual(w, o, 1);  // dense rows of the refinement's right-hand side
  PCU_PFOR(i, 0, m) {           // r' = S delta
    double v = 0.0;
#pragma unroll 1
    for (int j = 0; j < q; j++) v += w[o.S + i + ld * (c + j)] * alpha2[c + j];
    w[o.r + i] = v;
  }
  PCU_SYNC();
  pcu_dense_step(w, o, 1, alpha2, scratch);
  PCU_PFOR(j, 0, m) alpha[j] += alpha2[j];
  PCU_SYNC();
}
