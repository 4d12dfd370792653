// pcu_ip.cuh -- host-side interior-point driver (ParOptInteriorPoint mirror).
#pragma once

#include <algorithm>
#include <string>
#include <vector>

#include "pcu_kernels.cuh"
#include "pcu_problem.cuh"

// Options of ParOptInteriorPoint::addDefaultOptions (IP.cpp:536-727) that act on
// the hot path, same names and defaults.
struct IPOptions {
  double max_bound_value = 1e20;
  double abs_res_tol = 1e-6;
  double rel_func_tol = 0.0;
  double abs_step_tol = 0.0;
  double init_barrier_param = 0.1;
  double penalty_gamma = 1000.0;
  double penalty_descent_fraction = 0.3;
  double min_rho_penalty_search = 0.0;
  double init_rho_penalty_search = 0.0;
  double armijo_constant = 1e-5;
  double monotone_barrier_fraction = 0.25;
  double monotone_barrier_power = 1.1;
  double rel_bound_barrier = 1.0;
  double min_fraction_to_boundary = 0.95;
  double qn_sigma = 0.0;
  double function_precision = 1e-10;
  double design_precision = 1e-14;
  double start_affine_multiplier_min = 1.0;
  int use_line_search = 1;
  int use_backtracking_alpha = 0;
  int sequential_linear_method = 0;
  int use_quasi_newton_update = 1;
  int qn_subspace_size = 10;
  int max_major_iters = 5000;
  int max_line_iters = 10;
  int iterative_refinement_steps = 1;
  int hessian_reset_freq = 1000000;
  int output_level = 0;
  int write_output_frequency = 10;
  int history_level = 1;  // 0 none, 1 scalars, 2 + state checksums (one extra pass)
  // inexact-Newton GMRES path (IP.cpp:593-611, 639, 646, 668)
  int use_hvec_product = 0;
  // the problem's diagonal Hessian of the Lagrangian (evalHessianDiag) in place of the
  // quasi-Newton approximation (IP.cpp:1464, 1842, 3811, 4458)
  int use_diag_hessian = 0;
  int use_qn_gmres_precon = 1;
  int gmres_subspace_size = 0;
  double nk_switch_tol = 1e-3;
  double eisenstat_walker_alpha = 1.5;
  double eisenstat_walker_gamma = 1.0;
  double max_gmres_rtol = 0.1;
  double gmres_atol = 1e-30;
  std::string qn_type = "bfgs";
  std::string qn_update_type = "skip_negative_curvature";
  std::string qn_diag_type = "yty_over_yts";
  std::string norm_type = "infinity";
  std::string barrier_strategy = "monotone";
  std::string starting_point_strategy = "affine_step";
  std::string output_file;  // empty: no text log
  std::string ip_checkpoint_file;  // empty: no checkpoint (ParOptOptimizer.cpp:98)
  std::string problem_name;
};

// dst takes src's values; src's values are undefined afterwards.  Two vectors of the
// optimizer's own exchange their buffers (no copy), so that every handle keeps its
// identity; anything else is copied.
static inline int pcu_vec_take(pcu_vec *dst, pcu_vec *src) {
  if (dst->owns && src->owns && dst->managed == src->managed && dst->n == src->n &&
      dst->ctx == src->ctx) {
    std::swap(dst->d, src->d);
    std::swap(dst->host_touched, src->host_touched);
    return 0;
  }
  return pcu_vec_copy(dst, src);
}

struct Vars {  // ParOptVars (IP.h:373-389)
  pcu_vec *v[8] = {nullptr, nullptr, nullptr, nullptr,
                   nullptr, nullptr, nullptr, nullptr};
  std::vector<double> z, s, t, zs, zt;
  DVars dv() const {
    DVars d;
    d.x = v[PCU_X]->d;
    d.zl = v[PCU_ZL]->d;
    d.zu = v[PCU_ZU]->d;
    d.zw = v[PCU_ZW]->d;
    d.sw = v[PCU_SW]->d;
    d.tw = v[PCU_TW]->d;
    d.zsw = v[PCU_ZSW]->d;
    d.ztw = v[PCU_ZTW]->d;
    return d;
  }
};

// Compact limited-memory quasi-Newton approximations (ParOptLBFGS, ParOptLSR1;
// QN.cpp) with the vectors on the device and the small matrices on the host.
struct QuasiNewton {
  pcu_ctx *ctx = nullptr;
  int n = 0;
  int type = 0;  // 0 L-BFGS, 1 L-SR1
  int msub_max = 0, msub = 0;
  int damped = 0;
  int diag_yts_over_sts = 0;
  int fused_sr1 = 1;  // L-SR1: Z rebuild + stored-pair dots in one sweep (PCU_NO_FUSED_SR1: off)
  double b0 = 1.0;
  double eps = 1e-12;
  std::vector<pcu_vec *> S, Y, Zs;
  pcu_vec *r = nullptr;
  std::vector<double> D, L, B, M, d0, Mf;
  std::vector<double> piv;  // pivots of Mf, as doubles (the dense buffer's format)

  ~QuasiNewton();
  int init(pcu_ctx *c, int nvars, int kind, int m);
  void reset();
  int max_size() const { return type == 0 ? 2 * msub_max : msub_max; }
  int size() const { return type == 0 ? 2 * msub : msub; }
  void z_table(ColTable &t, int off) const;
  // kap = d0 * M^-1 * (d0 * rz)   (QN.cpp:398-412)
  void solve_compact(const double *rz, double *kap) const;
  int mult(pcu_vec *x, pcu_vec *y);
  int update(pcu_vec *s, pcu_vec *y, double yTy, double yTs, double sTs,
             const double *sZ, int *update_type, int steal = 0);
  void mat_update();
};

struct HistRec {
  double f[PCU_HIST_FIELDS];
  std::vector<double> dense;  // c, z, s, t, zs, zt
  std::string info;
};

struct IterTime {
  double total_ms = 0.0, callback_ms = 0.0, kkt_ms = 0.0;
};

struct StepScale {
  double alpha_x, alpha_z;
  int ceq;
  double m0, dm0, pnorm2;
};

struct pcu_ip {
  pcu_problem *prob = nullptr;
  pcu_ctx *ctx = nullptr;
  IPOptions opt;
  int nvars = 0, ncon = 0, nwcon = 0;
  WDesc wd;
  Vars variables, residual, update, refine;
  pcu_vec *lb = nullptr, *ub = nullptr, *g = nullptr;
  std::vector<pcu_vec *> Ac;
  pcu_vec *Dinv = nullptr, *Cw = nullptr;
  pcu_vec *d1 = nullptr, *d2 = nullptr, *t1 = nullptr;  // KKT-solve scratch
  pcu_vec *s_qn = nullptr, *y_qn = nullptr;
  pcu_vec *rx = nullptr, *rsw = nullptr, *rtw = nullptr;  // line-search trial
  // the multipliers of a first trial taken by TrialUpdateF (created on its first use)
  pcu_vec *rzl = nullptr, *rzu = nullptr, *rzw = nullptr, *rzsw = nullptr, *rztw = nullptr;
  pcu_vec *hdiag = nullptr;  // use_diag_hessian: h of the last gradient evaluation
  // g - A z at the current point, written by the last update pass (ncon >= 3): the first
  // pass of the next KKT solve reads it instead of g and the ncon constraint gradients
  pcu_vec *gaz = nullptr;
  int gaz_valid = 0;
  // A p_z of the iteration's two solves (first solve / its one refinement), written by the
  // pass-2 kernels while they read the constraint gradients anyway: with g - A z they give
  // the update pass -(g - A z+) without another sweep over the ncon columns.
  // apz_state: 0 nothing, 1 first solve there, 3 both there, -1 a solve did not report
  pcu_vec *apz1 = nullptr, *apz2 = nullptr;
  int apz_state = 0;
  // which of the two a pass-2 launch of this solve writes (null: none); `supported`: the
  // kernel about to run can emit it
  double *apz_target(int accumulate, bool supported);
  void apz_done(int accumulate, double *target);
  std::vector<double> c;
  double fobj = 0.0;
  std::vector<double> gamma_s, gamma_t;
  int gamma_custom = 0;  // set through setPenaltyGamma(const double*): not refreshed from the option
  QuasiNewton *qn = nullptr;
  int qn_external = 0;  // qn belongs to a pcu_qn handle (setQuasiNewton, IP.cpp:1193): not owned
  std::string qn_built_type;
  int qn_built_size = -1;

  double b0_used = 0.0;

  double barrier_param = 0.1, rho_penalty_search = 0.0;
  int niter = 0, neval = 0, ngeval = 0, nhvec = 0;
  int status = 0;
  std::vector<pcu_vec *> gmres_W;  // Krylov vectors (x block), gmres_subspace_size + 1

  // statistics of the last ResF launch
  double res_sums[11], res_max[5], res_min[2];
  double res_mu = 0.0;   // barrier of the last ResF launch
  int res_has_step = 0;  // the last ResF launch included the step terms
  int res_skip_hessian = 0;  // computeKKTRes with a step: leave the B p term to the caller
  double last_comp = 0.0;
  int force_direct_dots = 0;  // debugging: recompute [A|Z]^T p with multi-dots
  int opt_no_rhsgram = 0;     // debugging: keep the first solve's pass 1 out of the Gram pass
  int opt_no_fuse2s = 0;      // debugging: keep the step statistics in their own pass
  int stats_ready = 0;        // Pass2SF / Pass2SVF left the step statistics in stats_out
  double stats_tau_used = 0.0;
  double stats_out[32];
  double stats_hp2 = 0.0;     // sum h p^2 of the last Pass2SVHF (use_diag_hessian)
  int opt_no_wide = 0;        // debugging: more than 32 columns stay on the register-fed pass 2
  int opt_no_fuse21 = 0;      // debugging: refine elementwise, pass 2 and the next pass 1 separate
  // residual statistics of the NEXT iteration taken by the update passes (ResF layout)
  double upd_sums[11], upd_max[5], upd_min[2];
  int upd_stats_valid = 0;
  int opt_no_updstats = 0;    // debugging (PCU_NO_UPDSTATS): always run the residual pass
  int opt_no_trialupd = 0;    // debugging (PCU_NO_TRIALUPD): first trial by TrialF, then Update1FT
  int checkpoint_failed = 0;
  int opt_force_chain = 0;    // PCU_CHAIN=1: device chain also across GPUs
  int opt_no_gaz = 0;         // debugging (PCU_NO_GAZ): the update pass does not leave g - A z
  int opt_no_chain = 0;       // debugging (PCU_NO_CHAIN): dense algebra of the KKT solve on the host
  // The dense state of the KKT solve (pcu_dense.cuh): its inputs, the Gram matrix of
  // V = [A | Z], G and Ce with their LU factors.  dense_host (pinned) holds it in the
  // layout dense_off of the last setUpKKTSystem / kktChain; dense_dev is the work buffer
  // of pcu_dense_kernel.
  DenseOff dense_off = DenseOff();
  double *dense_dev = nullptr, *dense_host = nullptr;
  int dense_cap = 0;
  int denseReserve(const DenseOff &o);
  void densePack(const DenseOff &o, const Vars &vars, double mu, const double *gdiag);
  // quasi-Newton columns of a solve with the factors of the last setup: that setup's, or
  // none with use_qn = 0 or after a reset
  int denseWidth(int use_qn) const {
    return (qn && use_qn) ? std::min(dense_off.q, qn->size()) : 0;
  }
  int pass1_ready = 0;        // Pass2R1F left d1', d2' and [A|Z]^T t1' for the next solve
  std::vector<double> pass1_r;
  double stats_pmax = 0.0;  // |px|_inf of the last StatsF launch

  // resumable major loop state (locals of optimize(), IP.cpp:4570-4606)
  struct LoopState {
    int k = 0;
    int started = 0, finished = 0;
    int barrier_strategy = 0, input_barrier_strategy = 0;
    double fobj_prev = 0.0, alpha_prev = 0.0, alpha_xprev = 0.0, alpha_zprev = 0.0;
    double dm0_prev = 0.0, res_norm_prev = 0.0;
    int no_merit_function_improvement = 0, line_search_test = 0,
        line_search_failed = 0;
    // the last line search rejected its first trial: the next one takes it with TrialF
    // instead of the update pass, whose work would be lost again
    int first_trial_rejected = 0;
    std::string info;
    double last_pnorm2 = 0.0;
  } ls;

  std::vector<HistRec> history;
  std::vector<IterTime> times;
  FILE *outfp = nullptr;
  // Device timing of a major iteration (whole iteration, KKT solve, callbacks): two
  // event sets used alternately, so that iteration k is read out during iteration
  // k + 1 (after its first reduction has synchronised anyway) instead of costing a
  // synchronisation of its own.
  struct IterEvents {
    cudaEvent_t it0 = nullptr, it1 = nullptr, k0 = nullptr, k1 = nullptr;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t> > cb;
    size_t cb_used = 0;
    bool pending = false;
  } evs[2];
  int ev_cur = 0;
  int collect_times(IterEvents &e);  // waits for e.it1 when it is still pending
  int flush_times();

  ~pcu_ip();
  int init(pcu_problem *p);
  IPConst kconst() const;
  int norm_type_id() const;
  int ensure_qn();
  void refresh_penalties();

  // callbacks with device timing
  int cb_begin();
  int cb_end();
  double cb_collect();
  int evalObjCon(pcu_vec *x);
  int evalObjConGradient(pcu_vec *x, int same_point = 0);

  // hot-path functions (same names as the reference's private methods)
  int initAndCheckDesignAndBounds();
  int computeKKTRes(Vars &vars, double mu, Vars &res, Vars *step,
                    const double *ATp, const double *ZTp, int store = 1);
  void computeResNorm(Vars &res, double *max_prime, double *max_dual,
                      double *max_infeas, double *res_norm);
  // infinity-norm residual norms at another barrier value from the statistics
  // of the last (step-free) ResF launch; returns 0 when not available
  int resNormAtBarrier(Vars &vars, double mu, Vars &res, double *max_prime,
                       double *max_dual, double *max_infeas, double *res_norm);
  double compFromStats(Vars &vars);
  int setUpKKTDiagSystem(Vars &vars, int use_qn, int identity);
  int setUpKKTDiagRhs(Vars &vars, int use_qn, double mu);
  int setUpKKTSystem(Vars &vars, int use_qn, const double *gdiag, int with_rhs = 0);
  int kktChain(Vars &vars, Vars &b, Vars &y, int use_qn, double mu, double tau, double *VTp,
               int on_device);
  int computeKKTStep(Vars &vars, Vars &res, Vars &step, int use_qn,
                     int accumulate, double *VTp, int emit_res, double mu_res,
                     int *emitted, int rhs_from_vars = 0, double stats_tau = -1.0);
  void denseResidual(Vars &vars, double mu, Vars &res, Vars *step,
                     const double *ATp);
  int addMehrotraCorrectorResidual(Vars &step, Vars &res);
  int stepStats(Vars &vars, Vars &step, double tau, double *sums, double *mins);
  int scaleAndMerit(Vars &v, Vars &upd, double tau, double comp,
                    const double *VTp, double fixed_scale, StepScale *out,
                    int inexact_newton_step = 0);
  // computeKKTGMRESStep (IP.cpp:5789-6191): > 0 iterations taken, < 0 the step failed
  // the descent tests, 0 nothing done; *rc_err != 0 on a CUDA / callback error
  int computeKKTGMRESStep(Vars &vars, Vars &res, Vars &step, double rtol, double atol,
                          int use_qn, double *VTp, int *rc_err);
  int evalHvecProduct(pcu_vec *px, pcu_vec *hvec);
  int initLeastSquaresMultipliers();
  int initAffineStepMultipliers();
  int diagHessianRefused();  // use_diag_hessian with a route it does not cover: prints why
  int begin();
  int iterate_once(int *converged);
  int snapshot(int k, double comp, double max_prime, double max_dual,
               double max_infeas, double res_norm);
  void log_line(int k, double comp, double max_prime, double max_infeas,
                double max_dual);
};
