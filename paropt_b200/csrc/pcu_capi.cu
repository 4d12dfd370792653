// pcu_capi.cu -- extern "C" entry points of the interior-point optimizer
// (include/paropt_b200.h).  Context / vector / problem entry points live next to
// their implementations (pcu_vec.cu, pcu_problems.cu).
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "pcu_ip.cuh"

int pcu_mdot_enqueue(pcu_ctx *ctx, const double *x, const ColTable &cols,
                     int ncols, long long n, int dst_off);

namespace {

struct OptEntry {
  const char *name;
  int type;  // 0 float, 1 int/bool, 2 string/enum
  size_t offset;
  double lo, hi;  // numeric range (IP.cpp:536-727)
  const char *choices;  // '|'-separated enum values, or null
};

#define OPT_F(n, lo, hi) {#n, 0, offsetof(IPOptions, n), lo, hi, nullptr}
#define OPT_I(n, lo, hi) {#n, 1, offsetof(IPOptions, n), lo, hi, nullptr}
#define OPT_S(n, ch) {#n, 2, offsetof(IPOptions, n), 0, 0, ch}

const OptEntry OPTIONS[] = {
    OPT_F(max_bound_value, 0.0, 1e300),
    OPT_F(abs_res_tol, 0.0, 1e20),
    OPT_F(rel_func_tol, 0.0, 1e20),
    OPT_F(abs_step_tol, 0.0, 1e20),
    OPT_F(init_barrier_param, 0.0, 1e20),
    OPT_F(penalty_gamma, 0.0, 1e20),
    OPT_F(penalty_descent_fraction, 1e-6, 1.0),
    OPT_F(min_rho_penalty_search, 0.0, 1e20),
    OPT_F(init_rho_penalty_search, 0.0, 1e20),
    OPT_F(armijo_constant, 0.0, 1.0),
    OPT_F(monotone_barrier_fraction, 0.0, 1.0),
    OPT_F(monotone_barrier_power, 1.0, 10.0),
    OPT_F(rel_bound_barrier, 0.0, 1e20),
    OPT_F(min_fraction_to_boundary, 0.0, 1.0),
    OPT_F(qn_sigma, 0.0, 1e20),
    OPT_F(function_precision, 0.0, 1.0),
    OPT_F(design_precision, 0.0, 1.0),
    OPT_F(start_affine_multiplier_min, 0.0, 1e20),
    OPT_I(use_line_search, 0, 1),
    OPT_I(use_backtracking_alpha, 0, 1),
    OPT_I(sequential_linear_method, 0, 1),
    OPT_I(use_quasi_newton_update, 0, 1),
    OPT_I(qn_subspace_size, 0, 1000),
    OPT_I(max_major_iters, 0, 1000000),
    OPT_I(max_line_iters, 1, 100),
    OPT_I(iterative_refinement_steps, 0, 10),
    OPT_I(hessian_reset_freq, 1, 1000000),
    OPT_I(output_level, 0, 1000000),
    OPT_I(write_output_frequency, 0, 1000000),
    OPT_I(history_level, 0, 2),
    OPT_I(use_hvec_product, 0, 1),
    OPT_I(use_diag_hessian, 0, 1),
    OPT_I(use_qn_gmres_precon, 0, 1),
    OPT_I(gmres_subspace_size, 0, 1000),
    OPT_F(nk_switch_tol, 0.0, 1e20),
    OPT_F(eisenstat_walker_alpha, 0.0, 2.0),
    OPT_F(eisenstat_walker_gamma, 0.0, 1.0),
    OPT_F(max_gmres_rtol, 0.0, 1.0),
    OPT_F(gmres_atol, 0.0, 1.0),
    // The choices are the reference's own (IP.cpp:694-707), with the reference's own
    // behaviour: ParOptInteriorPoint's constructor builds a quasi-Newton object for "bfgs"
    // and "sr1" only ("scaled_bfgs" leaves qn = NULL exactly like "none", IP.cpp:262-277:
    // ParOptScaledQuasiNewton is created by ParOptOptimizer and handed in through
    // setQuasiNewton), and ParOptLBFGS / ParOptLSR1 test the diagonal type against
    // PAROPT_YTS_OVER_STS alone (QN.cpp:200, 256, 645): both "inner_*" values act as
    // "yty_over_yts".  Same option dictionary, same optimizer behaviour.
    OPT_S(qn_type, "bfgs|scaled_bfgs|sr1|none"),
    OPT_S(qn_update_type, "skip_negative_curvature|damped_update"),
    OPT_S(qn_diag_type,
          "yty_over_yts|yts_over_sts|inner_yty_over_yts|inner_yts_over_sts"),
    OPT_S(norm_type, "infinity|l1|l2"),
    OPT_S(barrier_strategy,
          "monotone|mehrotra|mehrotra_predictor_corrector|complementarity_fraction"),
    OPT_S(starting_point_strategy,
          "least_squares_multipliers|affine_step|no_start_strategy"),
    OPT_S(output_file, nullptr),
    OPT_S(ip_checkpoint_file, nullptr),
    OPT_S(problem_name, nullptr),
};

const OptEntry *find_option(const char *name) {
  for (const OptEntry &e : OPTIONS)
    if (strcmp(e.name, name) == 0) return &e;
  return nullptr;
}

bool in_choices(const char *choices, const char *value) {
  std::string all(choices);
  size_t pos = 0;
  while (pos <= all.size()) {
    size_t next = all.find('|', pos);
    if (next == std::string::npos) next = all.size();
    if (all.compare(pos, next - pos, value) == 0 && strlen(value) == next - pos)
      return true;
    pos = next + 1;
  }
  return false;
}

Vars *bundle(pcu_ip *ip, int which) {
  switch (which) {
    case PCU_VARS: return &ip->variables;
    case PCU_RESIDUAL: return &ip->residual;
    case PCU_UPDATE: return &ip->update;
    case PCU_REFINE: return &ip->refine;
  }
  return nullptr;
}

// [A | Z]^T x for a bundle's x component (direct multi-dot)
int step_dots(pcu_ip *ip, Vars &step, std::vector<double> &out) {
  const int qa = ip->qn ? ip->qn->size() : 0;
  out.assign(ip->ncon + qa + 1, 0.0);
  ColTable V;
  for (int j = 0; j < ip->ncon; j++) V.p[j] = ip->Ac[j]->d;
  if (qa > 0) ip->qn->z_table(V, ip->ncon);
  if (ip->ncon + qa == 0) return 0;
  if (pcu_mdot_enqueue(ip->ctx, step.v[PCU_X]->d, V, ip->ncon + qa, ip->nvars, 0))
    return 1;
  return ip->ctx->big_fetch(ip->ncon + qa, out.data());
}

}  // namespace

extern "C" {

pcu_ip *pcu_ip_create(pcu_problem *prob) {
  if (!prob) return nullptr;
  pcu_ip *ip = new pcu_ip;
  if (ip->init(prob)) {
    delete ip;
    return nullptr;
  }
  return ip;
}

void pcu_ip_destroy(pcu_ip *ip) {
  if (!ip) return;
  cudaStreamSynchronize(ip->ctx->stream);
  delete ip;
}

int pcu_ip_set_option_float(pcu_ip *ip, const char *name, double value) {
  const OptEntry *e = find_option(name);
  if (!e) return 1;
  if (e->type == 1) return pcu_ip_set_option_int(ip, name, (int)value);
  if (e->type != 0 || value < e->lo || value > e->hi) return 1;
  *(double *)((char *)&ip->opt + e->offset) = value;
  return 0;
}

int pcu_ip_set_option_int(pcu_ip *ip, const char *name, int value) {
  const OptEntry *e = find_option(name);
  if (!e) return 1;
  if (e->type == 0) return pcu_ip_set_option_float(ip, name, (double)value);
  if (e->type != 1 || value < e->lo || value > e->hi) return 1;
  *(int *)((char *)&ip->opt + e->offset) = value;
  return 0;
}

int pcu_ip_set_option_str(pcu_ip *ip, const char *name, const char *value) {
  const OptEntry *e = find_option(name);
  if (!e || e->type != 2 || !value) return 1;
  if (e->choices && !in_choices(e->choices, value)) return 1;
  *(std::string *)((char *)&ip->opt + e->offset) = value;
  return 0;
}

int pcu_ip_begin(pcu_ip *ip) { return ip->begin(); }

int pcu_ip_iterate(pcu_ip *ip, int max_iters, int *converged) {
  int conv = 0;
  ip->upd_stats_valid = 0;  // the caller may have touched the state between calls
  for (int i = 0; i < max_iters && !conv; i++) {
    if (ip->ls.k >= ip->opt.max_major_iters) break;
    if (ip->iterate_once(&conv)) return 1;
  }
  if (converged) *converged = conv;
  return ip->flush_times();
}

int pcu_ip_optimize(pcu_ip *ip) {
  if (ip->begin()) return 1;
  int conv = 0;
  while (!conv && ip->ls.k < ip->opt.max_major_iters) {
    if (ip->iterate_once(&conv)) return 1;
  }
  return ip->flush_times();
}

// resetDesignAndBounds (IP.cpp:1249-1251)
int pcu_ip_reset_design_and_bounds(pcu_ip *ip) {
  if (!ip) return 1;
  return ip->prob->getVarsAndBounds(ip->variables.v[PCU_X], ip->lb, ip->ub);
}

// setPenaltyGamma(double) (IP.cpp:1128-1153): every dense and sparse penalty
int pcu_ip_set_penalty_gamma(pcu_ip *ip, double gamma) {
  if (!ip) return 1;
  if (gamma >= 0.0) {
    ip->opt.penalty_gamma = gamma;
    ip->gamma_custom = 0;
    ip->refresh_penalties();
  }
  return 0;
}

// setPenaltyGamma(const double*) (IP.cpp:1160-1173): dense constraints only,
// negative entries keep their value
int pcu_ip_set_penalty_gamma_array(pcu_ip *ip, const double *gamma) {
  if (!ip || (!gamma && ip->ncon > 0)) return 1;
  ip->refresh_penalties();
  for (int i = 0; i < ip->ncon; i++) {
    if (gamma[i] >= 0.0) {
      ip->gamma_s[i] = i < ip->prob->ninequality ? 0.0 : gamma[i];
      ip->gamma_t[i] = gamma[i];
    }
  }
  ip->gamma_custom = 1;
  return 0;
}

int pcu_ip_get_penalty_gamma(pcu_ip *ip, double *gamma_t) {
  if (!ip) return 1;
  ip->refresh_penalties();
  for (int i = 0; i < ip->ncon; i++) gamma_t[i] = ip->gamma_t[i];
  return 0;
}

// resetProblemInstance (IP.cpp:745-764)
int pcu_ip_reset_problem(pcu_ip *ip, pcu_problem *prob) {
  if (!ip || !prob) return 1;
  const pcu_weighting &a = prob->weighting, &b = ip->prob->weighting;
  if (prob->ctx != ip->ctx || prob->nvars != ip->nvars || prob->ncon != ip->ncon ||
      prob->nwcon != ip->nwcon || prob->ninequality != ip->prob->ninequality ||
      prob->nwinequality != ip->prob->nwinequality || prob->use_lower != ip->prob->use_lower ||
      prob->use_upper != ip->prob->use_upper || a.nwcon != b.nwcon || a.wstart != b.wstart ||
      a.nw != b.nw || a.wstride != b.wstride || a.coef0 != b.coef0 ||
      a.coef_rest != b.coef_rest || a.wconst != b.wconst) {
    fprintf(stderr, "ParOpt: Incompatible problem instance\n");
    return 1;
  }
  ip->prob = prob;
  ip->gaz_valid = 0;
  return 0;
}

// resetQuasiNewtonHessian (IP.cpp:1241-1245)
int pcu_ip_reset_quasi_newton(pcu_ip *ip) {
  if (!ip) return 1;
  if (ip->qn) ip->qn->reset();
  return 0;
}

// ------------------------------------------------------------- checkpoint file
// Global offsets of this rank's slices (var_range / wcon_range, IP.cpp:214-229)
static int checkpoint_ranges(pcu_ip *ip, long long *n0, long long *ntot, long long *w0,
                             long long *wtot) {
  pcu_ctx *ctx = ip->ctx;
  std::vector<double> sizes(2 * (size_t)ctx->world, 0.0);
  sizes[2 * ctx->rank] = ip->nvars;
  sizes[2 * ctx->rank + 1] = ip->nwcon;
  if (pcu_ctx_allreduce_sum(ctx, sizes.data(), (int)sizes.size())) return 1;
  *n0 = *w0 = *ntot = *wtot = 0;
  for (int r = 0; r < ctx->world; r++) {
    if (r < ctx->rank) {
      *n0 += (long long)sizes[2 * r];
      *w0 += (long long)sizes[2 * r + 1];
    }
    *ntot += (long long)sizes[2 * r];
    *wtot += (long long)sizes[2 * r + 1];
  }
  return 0;
}

int pcu_ip_write_solution(pcu_ip *ip, const char *filename) {
  if (!ip || !filename) return 1;
  pcu_ctx *ctx = ip->ctx;
  long long n0, ntot, w0, wtot;
  if (checkpoint_ranges(ip, &n0, &ntot, &w0, &wtot)) return 1;
  const int c = ip->ncon;
  Vars &v = ip->variables;
  if (ctx->rank == 0) {  // header + dense parts (IP.cpp:902-917), file truncated
    FILE *fp = fopen(filename, "wb");
    if (!fp) return 1;
    const int sizes[3] = {(int)ntot, (int)wtot, c};
    fwrite(sizes, sizeof(int), 3, fp);
    fwrite(&ip->barrier_param, sizeof(double), 1, fp);
    const std::vector<double> *parts[5] = {&v.s, &v.t, &v.z, &v.zs, &v.zt};
    for (auto p : parts) fwrite(p->data(), sizeof(double), c, fp);
    fclose(fp);
  }
  double flag = 1.0;  // the other ranks write after the file exists
  if (pcu_ctx_allreduce_sum(ctx, &flag, 1)) return 1;
  FILE *fp = fopen(filename, "r+b");
  if (!fp) return 1;
  const long long base = 3 * (long long)sizeof(int) + (5LL * c + 1) * (long long)sizeof(double);
  std::vector<double> host((size_t)std::max(ip->nvars, ip->nwcon) + 1);
  int fail = 0;
  auto put = [&](pcu_vec *vec, long long off_elems, int count) {
    if (count == 0) return;
    if (pcu_vec_to_host(vec, host.data(), count)) fail = 1;
    if (fseeko(fp, (off_t)(base + off_elems * (long long)sizeof(double)), SEEK_SET) != 0) fail = 1;
    if (fwrite(host.data(), sizeof(double), count, fp) != (size_t)count) fail = 1;
  };
  put(v.v[PCU_X], n0, ip->nvars);
  put(v.v[PCU_ZL], ntot + n0, ip->nvars);
  put(v.v[PCU_ZU], 2 * ntot + n0, ip->nvars);
  if (wtot > 0) {
    put(v.v[PCU_ZW], 3 * ntot + w0, ip->nwcon);
    put(v.v[PCU_SW], 3 * ntot + wtot + w0, ip->nwcon);
  }
  fclose(fp);
  flag = fail;
  if (pcu_ctx_allreduce_sum(ctx, &flag, 1)) return 1;
  return flag != 0.0;
}

int pcu_ip_read_solution(pcu_ip *ip, const char *filename) {
  if (!ip || !filename) return 1;
  long long n0, ntot, w0, wtot;
  if (checkpoint_ranges(ip, &n0, &ntot, &w0, &wtot)) return 1;
  FILE *fp = fopen(filename, "rb");
  if (!fp) return 1;
  const int c = ip->ncon;
  Vars &v = ip->variables;
  int sizes[3] = {0, 0, 0};
  if (fread(sizes, sizeof(int), 3, fp) != 3 || sizes[0] != (int)ntot || sizes[1] != (int)wtot ||
      sizes[2] != c) {
    if (ip->ctx->rank == 0)
      fprintf(stderr, "ParOpt: Problem size incompatible with solution file\n");
    fclose(fp);
    return 1;
  }
  int fail = 0;
  // every rank reads the replicated dense parts itself (root + Bcast in the reference)
  if (fread(&ip->barrier_param, sizeof(double), 1, fp) != 1) fail = 1;
  std::vector<double> *parts[5] = {&v.s, &v.t, &v.z, &v.zs, &v.zt};
  for (auto p : parts)
    if (c > 0 && fread(p->data(), sizeof(double), c, fp) != (size_t)c) fail = 1;
  const long long base = 3 * (long long)sizeof(int) + (5LL * c + 1) * (long long)sizeof(double);
  std::vector<double> host((size_t)std::max(ip->nvars, ip->nwcon) + 1);
  auto get = [&](pcu_vec *vec, long long off_elems, int count) {
    if (count == 0) return;
    if (fseeko(fp, (off_t)(base + off_elems * (long long)sizeof(double)), SEEK_SET) != 0) fail = 1;
    if (fread(host.data(), sizeof(double), count, fp) != (size_t)count) fail = 1;
    if (pcu_vec_from_host(vec, host.data(), count)) fail = 1;
  };
  get(v.v[PCU_X], n0, ip->nvars);
  get(v.v[PCU_ZL], ntot + n0, ip->nvars);
  get(v.v[PCU_ZU], 2 * ntot + n0, ip->nvars);
  if (wtot > 0) {
    get(v.v[PCU_ZW], 3 * ntot + w0, ip->nwcon);
    get(v.v[PCU_SW], 3 * ntot + wtot + w0, ip->nwcon);
  }
  fclose(fp);
  ip->upd_stats_valid = 0;
  return fail;
}

int pcu_ip_get_point(pcu_ip *ip, pcu_vec **x, pcu_vec **zw, pcu_vec **zl,
                     pcu_vec **zu, pcu_vec **sw, pcu_vec **tw) {
  Vars &v = ip->variables;
  if (x) *x = v.v[PCU_X];
  if (zw) *zw = v.v[PCU_ZW];
  if (zl) *zl = v.v[PCU_ZL];
  if (zu) *zu = v.v[PCU_ZU];
  if (sw) *sw = v.v[PCU_SW];
  if (tw) *tw = v.v[PCU_TW];
  return 0;
}

int pcu_ip_get_dense(pcu_ip *ip, double *z, double *s, double *t, double *zs,
                     double *zt, double *c) {
  Vars &v = ip->variables;
  const size_t bytes = sizeof(double) * ip->ncon;
  if (z) memcpy(z, v.z.data(), bytes);
  if (s) memcpy(s, v.s.data(), bytes);
  if (t) memcpy(t, v.t.data(), bytes);
  if (zs) memcpy(zs, v.zs.data(), bytes);
  if (zt) memcpy(zt, v.zt.data(), bytes);
  if (c) memcpy(c, ip->c.data(), bytes);
  return 0;
}

double pcu_ip_barrier_param(pcu_ip *ip) { return ip->barrier_param; }

int pcu_ip_complementarity(pcu_ip *ip, double *comp) { return pcu_ip_comp(ip, comp); }

int pcu_ip_counters(pcu_ip *ip, int *niter, int *neval, int *ngeval) {
  if (niter) *niter = ip->niter;
  if (neval) *neval = ip->neval;
  if (ngeval) *ngeval = ip->ngeval;
  return 0;
}

int pcu_ip_status(pcu_ip *ip) { return ip->status; }

int pcu_ip_history_len(pcu_ip *ip) { return (int)ip->history.size(); }

int pcu_ip_history_get(pcu_ip *ip, int k, double *out, int out_len) {
  if (k < 0 || k >= (int)ip->history.size()) return 1;
  const HistRec &r = ip->history[k];
  const int need = PCU_HIST_FIELDS + (int)r.dense.size();
  if (out_len < need) return 1;
  memcpy(out, r.f, sizeof(double) * PCU_HIST_FIELDS);
  if (!r.dense.empty())
    memcpy(out + PCU_HIST_FIELDS, r.dense.data(), sizeof(double) * r.dense.size());
  return 0;
}

const char *pcu_ip_history_info(pcu_ip *ip, int k) {
  if (k < 0 || k >= (int)ip->history.size()) return "";
  return ip->history[k].info.c_str();
}

int pcu_ip_iter_times(pcu_ip *ip, int k, double *total_ms, double *callback_ms,
                      double *kkt_ms) {
  if (ip->flush_times()) return 1;
  if (k < 0 || k >= (int)ip->times.size()) return 1;
  if (total_ms) *total_ms = ip->times[k].total_ms;
  if (callback_ms) *callback_ms = ip->times[k].callback_ms;
  if (kkt_ms) *kkt_ms = ip->times[k].kkt_ms;
  return 0;
}

pcu_vec *pcu_ip_vars_vec(pcu_ip *ip, int which, int component) {
  Vars *b = bundle(ip, which);
  if (!b || component < 0 || component > 7) return nullptr;
  return b->v[component];
}

int pcu_ip_vars_dense_get(pcu_ip *ip, int which, double *out5c) {
  Vars *b = bundle(ip, which);
  if (!b) return 1;
  const int c = ip->ncon;
  const std::vector<double> *parts[5] = {&b->z, &b->s, &b->t, &b->zs, &b->zt};
  for (int k = 0; k < 5; k++) memcpy(out5c + k * c, parts[k]->data(), sizeof(double) * c);
  return 0;
}

int pcu_ip_vars_dense_set(pcu_ip *ip, int which, const double *in5c) {
  Vars *b = bundle(ip, which);
  if (!b) return 1;
  const int c = ip->ncon;
  std::vector<double> *parts[5] = {&b->z, &b->s, &b->t, &b->zs, &b->zt};
  for (int k = 0; k < 5; k++) memcpy(parts[k]->data(), in5c + k * c, sizeof(double) * c);
  ip->gaz_valid = 0;  // the multipliers z changed
  return 0;
}

pcu_vec *pcu_ip_state_vec(pcu_ip *ip, int id) {
  switch (id) {
    case 0: return ip->lb;
    case 1: return ip->ub;
    case 2: return ip->g;
    case 3: return ip->Dinv;
    case 4: return ip->Cw;
  }
  if (id >= 100 && id < 100 + ip->ncon) return ip->Ac[id - 100];
  return nullptr;
}

int pcu_ip_set_obj_con(pcu_ip *ip, double fobj, const double *c) {
  ip->fobj = fobj;
  for (int i = 0; i < ip->ncon; i++) ip->c[i] = c[i];
  return 0;
}

int pcu_ip_set_barrier(pcu_ip *ip, double mu, double rho) {
  ip->barrier_param = mu;
  ip->rho_penalty_search = rho;
  return 0;
}

int pcu_ip_qn_update(pcu_ip *ip, pcu_vec *s, pcu_vec *y, int *update_type) {
  if (ip->ensure_qn() || !ip->qn) return 1;
  double yy, ys, ss;
  if (pcu_vec_dot(y, y, &yy) || pcu_vec_dot(y, s, &ys) || pcu_vec_dot(s, s, &ss))
    return 1;
  int ut = 0;
  if (ip->qn->update(s, y, yy, ys, ss, nullptr, &ut)) return 1;
  if (update_type) *update_type = ut;
  return 0;
}

int pcu_ip_qn_reset(pcu_ip *ip) {
  if (ip->ensure_qn() || !ip->qn) return 1;
  ip->qn->reset();
  return 0;
}

int pcu_ip_qn_mult(pcu_ip *ip, pcu_vec *x, pcu_vec *y) {
  if (ip->ensure_qn() || !ip->qn) return 1;
  return ip->qn->mult(x, y);
}

int pcu_ip_qn_compact(pcu_ip *ip, double *b0, int *size, double *d0, double *M) {
  if (ip->ensure_qn() || !ip->qn) return 1;
  const int q = ip->qn->size();
  if (b0) *b0 = ip->qn->b0;
  if (size) *size = q;
  if (d0 && q > 0) memcpy(d0, ip->qn->d0.data(), sizeof(double) * q);
  if (M && q > 0) memcpy(M, ip->qn->M.data(), sizeof(double) * q * q);
  return 0;
}

int pcu_ip_kkt_res(pcu_ip *ip, int vars, double mu, int res) {
  Vars *v = bundle(ip, vars), *r = bundle(ip, res);
  if (!v || !r) return 1;
  if (ip->ensure_qn()) return 1;
  ip->refresh_penalties();
  return ip->computeKKTRes(*v, mu, *r, nullptr, nullptr, nullptr);
}

int pcu_ip_res_norm(pcu_ip *ip, double *max_prime, double *max_dual,
                    double *max_infeas, double *res_norm) {
  double a, b, c, d;
  ip->computeResNorm(ip->residual, &a, &b, &c, &d);
  if (max_prime) *max_prime = a;
  if (max_dual) *max_dual = b;
  if (max_infeas) *max_infeas = c;
  if (res_norm) *res_norm = d;
  return 0;
}

int pcu_ip_comp(pcu_ip *ip, double *comp) {
  // statistics of a residual pass written to the `refine` bundle (scratch)
  if (ip->ensure_qn()) return 1;
  ip->refresh_penalties();
  if (ip->computeKKTRes(ip->variables, ip->barrier_param, ip->refine, nullptr,
                        nullptr, nullptr))
    return 1;
  *comp = ip->compFromStats(ip->variables);
  return 0;
}

int pcu_ip_setup_kkt_diag(pcu_ip *ip, int use_qn) {
  if (ip->diagHessianRefused() || ip->ensure_qn()) return 1;
  if (ip->setUpKKTDiagSystem(ip->variables, use_qn, 0)) return 1;
  return ip->setUpKKTSystem(ip->variables, 0, nullptr);
}

int pcu_ip_setup_kkt(pcu_ip *ip, int use_qn) {
  if (ip->ensure_qn()) return 1;
  return ip->setUpKKTSystem(ip->variables, use_qn, nullptr);
}

int pcu_ip_kkt_step(pcu_ip *ip, int res, int step, int use_qn) {
  Vars *r = bundle(ip, res), *s = bundle(ip, step);
  if (!r || !s) return 1;
  return ip->computeKKTStep(ip->variables, *r, *s, use_qn, 0, nullptr, 0, 0.0, nullptr);
}

int pcu_ip_add_kkt_res_step(pcu_ip *ip, int step, int res) {
  Vars *s = bundle(ip, step), *r = bundle(ip, res);
  if (!r || !s) return 1;
  if (ip->diagHessianRefused() || ip->ensure_qn()) return 1;
  ip->refresh_penalties();
  std::vector<double> dots;
  if (step_dots(ip, *s, dots)) return 1;
  return ip->computeKKTRes(ip->variables, ip->barrier_param, *r, s, dots.data(),
                           dots.data() + ip->ncon);
}

int pcu_ip_kkt_solve(pcu_ip *ip, int res, int step, int on_device) {
  Vars *r = bundle(ip, res), *s = bundle(ip, step);
  if (!r || !s) return 1;
  if (ip->diagHessianRefused() || ip->ensure_qn()) return 1;
  if (on_device && !ip->ctx->chain_ok()) return 1;
  ip->refresh_penalties();
  const int m = ip->ncon + (ip->qn ? ip->qn->size() : 0);
  if (m < 1 || m > PCU_DENSE_MAXM) return 1;
  std::vector<double> vtp(m + 1);
  double tau = ip->opt.min_fraction_to_boundary;
  if (1.0 - ip->barrier_param >= tau) tau = 1.0 - ip->barrier_param;
  const int rc = ip->kktChain(ip->variables, *r, *s, 1, ip->barrier_param, tau, vtp.data(),
                              on_device);
  ip->stats_ready = 0;
  return rc;
}

int pcu_ip_max_step(pcu_ip *ip, double tau, int step, double *max_x,
                    double *max_z) {
  Vars *s = bundle(ip, step);
  if (!s) return 1;
  double sums[StatsF::NS], mins[2];
  if (ip->stepStats(ip->variables, *s, tau, sums, mins)) return 1;
  *max_x = mins[0];
  *max_z = mins[1];
  return 0;
}

int pcu_ip_comp_step(pcu_ip *ip, double ax, double az, int step, double *comp) {
  Vars *s = bundle(ip, step);
  if (!s) return 1;
  double c0;
  if (pcu_ip_comp(ip, &c0)) return 1;  // provides the global count
  double sums[StatsF::NS], mins[2];
  if (ip->stepStats(ip->variables, *s, 1.0, sums, mins)) return 1;
  Vars &v = ip->variables;
  double product = (sums[0] + ax * sums[1] + az * sums[2] + ax * az * sums[3]) /
                       ip->opt.rel_bound_barrier +
                   (sums[4] + ax * sums[5] + az * sums[6] + ax * az * sums[7]);
  double count = ip->res_sums[1];
  for (int i = 0; i < ip->ncon; i++) {
    product += (v.s[i] + ax * s->s[i]) * (v.zs[i] + az * s->zs[i]) +
               (v.t[i] + ax * s->t[i]) * (v.zt[i] + az * s->zt[i]);
    count += 2.0;
  }
  *comp = count != 0.0 ? product / count : 0.0;
  return 0;
}

int pcu_ip_merit_init_deriv(pcu_ip *ip, double max_x, double *merit,
                            double *pmerit) {
  if (ip->ensure_qn()) return 1;
  ip->refresh_penalties();
  std::vector<double> dots;
  if (step_dots(ip, ip->update, dots)) return 1;
  StepScale sc;
  if (ip->scaleAndMerit(ip->variables, ip->update, 1.0, 0.0, dots.data(), max_x, &sc))
    return 1;
  *merit = sc.m0;
  *pmerit = sc.dm0;
  return 0;
}

int pcu_ip_get_gram(pcu_ip *ip, double *G, double *Ce, int *q) {
  const DenseOff &o = ip->dense_off;  // (all zero before the first setup)
  const double *h = ip->dense_host;
  if (q) *q = o.q;
  if (G && h) memcpy(G, h + o.Graw, sizeof(double) * o.c * o.c);
  if (Ce && h) memcpy(Ce, h + o.Ceraw, sizeof(double) * o.q * o.q);
  return 0;
}

}  // extern "C"
