// pcu_problem.cuh -- the problem object behind pcu_problem (ParOptProblem).
#pragma once

#include <vector>

#include "pcu_ctx.cuh"

struct pcu_problem {
  pcu_ctx *ctx = nullptr;
  int nvars = 0, ncon = 0, nwcon = 0;
  int ninequality = 0, nwinequality = 0;
  int use_lower = 1, use_upper = 1;
  pcu_weighting weighting;
  // per-constraint constants of the weighting rows (W-sized), or null: weighting.wconst
  pcu_vec *wconst_vec = nullptr;
  double callback_ms = 0.0;  // device time inside the callbacks
  cudaEvent_t cb0 = nullptr, cb1 = nullptr;
  bool time_callbacks = true;
  // Set by the optimizer right before a callback: the vector handed over holds
  // bit-identical values to the one of the previous callback (the accepted
  // line-search trial point).  Host-array problems skip the device->host copy.
  int same_point_hint = 0;
  long long h2d_bytes = 0, d2h_bytes = 0;  // host-array problems only

  virtual ~pcu_problem() {}
  virtual int getVarsAndBounds(pcu_vec *x, pcu_vec *lb, pcu_vec *ub) = 0;
  // fobj / cons are host outputs (the reference's signature, ParOptProblem.h:157)
  virtual int evalObjCon(pcu_vec *x, double *fobj, double *cons) = 0;
  virtual int evalObjConGradient(pcu_vec *x, pcu_vec *g, pcu_vec **Ac) = 0;
  // optional hooks with the reference's empty defaults (ParOptProblem.cpp:220-223)
  virtual int qnUpdateCorrection(pcu_vec *, const double *, pcu_vec *, pcu_vec *, pcu_vec *) {
    return 0;
  }
  virtual bool hasQnUpdateCorrection() const { return false; }
  virtual int writeOutput(int, pcu_vec *) { return 0; }
  // hvec = H(x, z, zw) px, the Hessian of the Lagrangian (ParOptProblem.h:188); only the
  // inexact-Newton GMRES path calls it (use_hvec_product, IP.cpp:5973, 1461).  The
  // reference's default prints an error and returns 0 (ParOptProblem.cpp:205-212);
  // here a problem without the callback fails the step.
  virtual int evalHvecProduct(pcu_vec *, const double *, pcu_vec *, pcu_vec *, pcu_vec *) {
    return 1;
  }
  virtual bool hasHvecProduct() const { return false; }
  // h = the diagonal of the Hessian of the Lagrangian at (x, z, zw); the optimizer calls
  // it after every gradient evaluation when use_diag_hessian is set, and refuses that
  // option for a problem without it.
  virtual int evalHessianDiag(pcu_vec *, const double *, pcu_vec *, pcu_vec *) { return 1; }
  virtual bool hasHessianDiag() const { return false; }
};

WDesc pcu_make_wdesc(const pcu_weighting &w, int nvars);
int pcu_validate_weighting(const pcu_weighting *w, int nvars, int ncon, int ninequality,
                           int nwinequality, const char *who);
