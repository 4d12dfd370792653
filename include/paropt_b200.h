/*
  paropt_b200.h -- C ABI of the B200-native interior-point hot path.

  This is the drop-in boundary a ParOpt maintainer binds (INTEGRATION.md shows
  the C++ adapter classes).  Every entry point cites the reference interface it
  replaces; paths are relative to the reference's src/ directory and
  IP.cpp = ParOptInteriorPoint.cpp, QN.cpp = ParOptQuasiNewton.cpp,
  SM.cpp = ParOptSparseMat.cpp.

  Conventions (kept from the reference, SURVEY.md 8b):
    * plain C types only; sizes are int (local sizes, as in ParOptVec.h:96);
    * functions returning int return 0 on success; on failure a message is also
      printed to stderr (reference style, IP.cpp:4534-4537);
    * all calls are collective over the ranks of the context and must be made in
      the same order on every rank (one host thread per rank / GPU);
    * reductions return the GLOBAL value on every rank (ParOptVec.cpp:63-170);
    * there is no CPU fallback: every call needs a CUDA device.
*/
#ifndef PAROPT_B200_H
#define PAROPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pcu_ctx pcu_ctx;
typedef struct pcu_vec pcu_vec;
typedef struct pcu_problem pcu_problem;
typedef struct pcu_ip pcu_ip;

/* ------------------------------------------------------------------ context
   Replaces the MPI communicator every reference object carries
   (ParOptProblem.h:48 MPI_Comm; IP.cpp:198-229 rank/size/ranges).           */

/* Library version string. */
const char *pcu_version(void);

/* One context per process / GPU.  `device` is the CUDA ordinal. */
pcu_ctx *pcu_ctx_create(int device);
void pcu_ctx_destroy(pcu_ctx *ctx);

/* Multi-GPU: rank 0 obtains a 128-byte NCCL unique id, the host side ships it
   to the other ranks (torch.distributed broadcast), then every rank calls
   pcu_ctx_init_comm.  Replaces MPI_Init / MPI_Comm_rank / MPI_Comm_size.      */
int pcu_nccl_unique_id(unsigned char id128[128]);
int pcu_ctx_init_comm(pcu_ctx *ctx, const unsigned char id128[128], int rank,
                      int world_size);
int pcu_ctx_rank(pcu_ctx *ctx);
int pcu_ctx_size(pcu_ctx *ctx);
int pcu_ctx_sync(pcu_ctx *ctx); /* cudaStreamSynchronize on the ctx stream */
void *pcu_ctx_stream(pcu_ctx *ctx); /* cudaStream_t, for callers that enqueue */
/* Number of kernels of THIS library launched on the context since creation.  */
int64_t pcu_ctx_kernel_launches(pcu_ctx *ctx);
/* Launch tuning knobs (no reference counterpart; results are unchanged up to
   summation order): "prefetch", "max_blocks_per_sm", "no_tma_tile" (1: keep
   the fused passes on the register-fed kernel), "tma_groups", "tma_npw",
   "tma_min_tiles", "tma_grid".  Returns 0, or 1 for an unknown name.          */
int pcu_ctx_set_param(pcu_ctx *ctx, const char *name, int value);
/* Per-kernel device timing: enable = 1 starts bracketing every launch of this
   library with CUDA events on the launching stream, 2 also clears the totals,
   0 stops.  profile_get returns kernel name, accumulated ms and launch count. */
int pcu_ctx_profile(pcu_ctx *ctx, int enable);
int pcu_ctx_profile_count(pcu_ctx *ctx);
int pcu_ctx_profile_get(pcu_ctx *ctx, int index, char *name, int name_len,
                        double *ms, int64_t *count);
/* Device-side timing helpers (cudaEvent on the ctx stream), milliseconds.     */
int pcu_ctx_timer_start(pcu_ctx *ctx);
int pcu_ctx_timer_stop(pcu_ctx *ctx, double *ms);

/* ------------------------------------------------------------------ vectors
   ParOptVec / ParOptBasicVec (ParOptVec.h:53-98, ParOptVec.cpp:15-217).      */
pcu_vec *pcu_vec_create(pcu_ctx *ctx, int n);               /* ParOptVec.cpp:15 */
void pcu_vec_destroy(pcu_vec *v);                           /* ParOptVec.cpp:25 */
int pcu_vec_size(pcu_vec *v);                               /* getArray return  */
int pcu_vec_set(pcu_vec *v, double alpha);                  /* :32  set         */
int pcu_vec_zero(pcu_vec *v);                               /* :41  zeroEntries */
int pcu_vec_copy(pcu_vec *dst, pcu_vec *src);               /* :50  copyValues  */
int pcu_vec_norm(pcu_vec *v, double *out);                  /* :63  norm        */
int pcu_vec_maxabs(pcu_vec *v, double *out);                /* :87  maxabs      */
int pcu_vec_l1norm(pcu_vec *v, double *out);                /* :106 l1norm      */
int pcu_vec_dot(pcu_vec *x, pcu_vec *y, double *out);       /* :124 dot         */
int pcu_vec_mdot(pcu_vec *x, pcu_vec **vecs, int nvecs,
                 double *out);                              /* :152 mdot        */
int pcu_vec_scale(pcu_vec *v, double alpha);                /* :177 scale       */
int pcu_vec_axpy(pcu_vec *y, double alpha, pcu_vec *x);     /* :194 axpy        */
/* getArray (ParOptVec.cpp:211) is a host-pointer contract in the reference.
   Here the storage is device memory: device_ptr gives the raw pointer for
   GPU-resident callers, the two copies serve host callbacks.                  */
double *pcu_vec_device_ptr(pcu_vec *v);
int pcu_vec_to_host(pcu_vec *v, double *host, int n);   /* D2H, synchronous */
int pcu_vec_from_host(pcu_vec *v, const double *host, int n); /* H2D, sync  */
/* getArray for reference code that loops over raw pointers (the ~25 private
   methods of ParOptInteriorPoint, ParOptTrustRegion, user callbacks): a context
   with pcu_ctx_set_param(ctx, "managed_vectors", 1) allocates every vector in
   unified memory.  pcu_vec_host_ptr synchronises the context's stream and returns
   a pointer the host may read AND write; the vector is marked host-touched and is
   moved back to the device (prefetch on the context's stream) by the next library
   call that uses it, so no write through the pointer is ever lost.  Returns NULL
   for a device-only vector.                                                     */
double *pcu_vec_host_ptr(pcu_vec *v);
int pcu_vec_is_managed(pcu_vec *v);

/* ------------------------------------------------------------------ problem
   ParOptProblem (ParOptProblem.h:42-299).  The sparse "weighting" constraints
   are declared as data so that Aw, Aw^T and Aw D^-1 Aw^T fuse into the kernels
   (they replace the callbacks evalSparseCon / addSparseJacobian /
   addSparseJacobianTranspose / addSparseInnerProduct, ParOptProblem.h:225-272,
   and ParOptQuasiDefBlockMat, SM.cpp:11-229, with nwblock = 1):
       cw_i(x) = wconst + coef0 * x[j0] + coef_rest * sum_{k=1}^{nw-1} x[j0+k],
       j0 = wstart + i * wstride,  i < nwcon,  wstride >= nw.                  */
typedef struct pcu_weighting {
  int nwcon;      /* local number of weighting constraints (0 = none)          */
  int wstart;     /* first variable of constraint 0                            */
  int nw;         /* variables per constraint                                  */
  int wstride;    /* distance between first variables of consecutive rows      */
  double coef0;   /* coefficient of the first variable of a row                */
  double coef_rest; /* coefficient of the other nw-1 variables                 */
  double wconst;  /* constant term                                             */
} pcu_weighting;

/* Host/device callbacks: the exact callback set of ParOptProblem
   (getVarsAndBounds :143, evalObjCon :157, evalObjConGradient :172).  Vectors
   are pcu_vec handles; a host callback uses pcu_vec_to_host / _from_host, a
   GPU-resident one uses pcu_vec_device_ptr and enqueues on pcu_ctx_stream.    */
typedef struct pcu_problem_callbacks {
  void *user;
  int (*get_vars_and_bounds)(void *user, pcu_vec *x, pcu_vec *lb, pcu_vec *ub);
  int (*eval_obj_con)(void *user, pcu_vec *x, double *fobj, double *cons);
  int (*eval_obj_con_gradient)(void *user, pcu_vec *x, pcu_vec *g, pcu_vec **Ac);
  /* Optional (NULL = the reference's empty default, ParOptProblem.cpp:220-223):
     computeQuasiNewtonUpdateCorrection (ParOptProblem.h:287; called right before
     the quasi-Newton update, IP.cpp:4258; z = ncon host doubles) and writeOutput
     (ParOptProblem.h:296; called every write_output_frequency iterations at the
     top of the major loop, IP.cpp:4620-4631).                                  */
  int (*qn_update_correction)(void *user, pcu_vec *x, const double *z, pcu_vec *zw,
                              pcu_vec *s, pcu_vec *y);
  int (*write_output)(void *user, int iter, pcu_vec *x);
  /* Optional: hvec = H(x, z, zw) px, the Hessian of the Lagrangian
     (ParOptProblem::evalHvecProduct, ParOptProblem.h:188).  Needed only with the option
     use_hvec_product (inexact-Newton GMRES steps, IP.cpp:4853-4900, 5789-6191); NULL
     makes such a step fail.                                                      */
  int (*eval_hvec_product)(void *user, pcu_vec *x, const double *z, pcu_vec *zw,
                           pcu_vec *px, pcu_vec *hvec);
} pcu_problem_callbacks;

/* ParOptProblem::setProblemSizes / setNumInequalities (ParOptProblem.cpp:47-76)
   nvars, nwcon are LOCAL sizes; ncon is global.                               */
pcu_problem *pcu_problem_create(pcu_ctx *ctx, int nvars, int ncon,
                                int ninequality, int nwinequality,
                                int use_lower, int use_upper,
                                const pcu_weighting *weighting,
                                const pcu_problem_callbacks *callbacks);
void pcu_problem_destroy(pcu_problem *prob);

/* ---- ParOptQuasiDefMat / ParOptQuasiDefBlockMat as a stand-alone object ------
   (ParOptSparseMat.h:18-104, nwblock = 1; ParOptSparseMat.cpp:41-224).  What
   ParOptProblem::createQuasiDefMat() returns for a problem whose sparse
   constraints are the weighting rows of a pcu_weighting descriptor.
     factor(x, Dinv, Cdiag)  Ew = Cdiag + Aw Dinv Aw^T, inverted; 0 = ok, k > 0 =
                             zero pivot in (local) row k - 1, < 0 = bad arguments.
                             Dinv is kept by reference until the next factor().
     apply3(bx, yx, yw)      [[D, Aw^T], [Aw, -C]] [yx; -yw] = [bx; 0]
     apply4(bx, bw, yx, yw)  ... = [bx; bw]   (inputs unmodified)                */
typedef struct pcu_blockmat pcu_blockmat;
pcu_blockmat *pcu_blockmat_create(pcu_ctx *ctx, int nvars, const pcu_weighting *weighting);
void pcu_blockmat_destroy(pcu_blockmat *mat);
int pcu_blockmat_factor(pcu_blockmat *mat, pcu_vec *x, pcu_vec *Dinv, pcu_vec *Cdiag);
int pcu_blockmat_apply3(pcu_blockmat *mat, pcu_vec *bx, pcu_vec *yx, pcu_vec *yw);
int pcu_blockmat_apply4(pcu_blockmat *mat, pcu_vec *bx, pcu_vec *bw, pcu_vec *yx,
                        pcu_vec *yw);

/* Block form, nwblock > 1 (ParOptQuasiDefBlockMat with nwblock = nb, SM.cpp:72-111,
   196-224): the sparse constraints come in groups of nb consecutive rows that share
   the nw variables of one block; block b covers the variables
   [wstart + b * wstride, + nw), its rows are  cw_{b nb + r}(x) = wconst[r] +
   sum_k coef[r * nw + k] * x[wstart + b * wstride + k].  Ew = Cdiag + Aw Dinv Aw^T is
   then block diagonal with dense nb x nb blocks, kept packed upper and factored by
   Cholesky (LAPACK dpptrf / dpptrs "U" in the reference).  1 <= nb <= 8, nw <= 64;
   coef / wconst are copied.  factor / apply3 / apply4 as for pcu_blockmat_create;
   factor returns k > 0 when the block holding (local) row k - 1 is not positive
   definite.                                                                       */
typedef struct pcu_block_weighting {
  int nblocks;        /* local number of blocks (nwcon = nblocks * nb)              */
  int wstart;         /* first variable of block 0                                  */
  int nw;             /* variables per block                                        */
  int wstride;        /* distance between the first variables of consecutive blocks */
  int nb;             /* constraints per block = nwblock                            */
  const double *coef; /* [nb][nw] row-major                                         */
  const double *wconst; /* [nb], may be NULL (zeros)                                */
} pcu_block_weighting;
pcu_blockmat *pcu_blockmat_create_blocks(pcu_ctx *ctx, int nvars,
                                         const pcu_block_weighting *blocks);

/* ---- ParOptQuasiDefSparseMat (ParOptSparseMat.cpp:231-451): the quasi-definite matrix
   of a problem whose sparse constraints are a general CSR Jacobian A (nwcon x nvars,
   rank-local: ParOptSparseProblem, ParOptProblem.h:301-407).  What createQuasiDefMat()
   returns for such a problem.
     create      pattern rowp[nwcon + 1], cols[nnz] (host; any column order inside a row, no
                 duplicates); symbolic Cholesky of K = C + A D^-1 A^T on the host.
                 ordering: 0 natural, 1 minimum degree.  ctx may be NULL: symbolic data
                 only (pcu_sparsemat_symbolic / _info), no device calls.
     set_data    the nnz Jacobian values in CSR order (host array; what
                 getSparseJacobianData returns after evalSparseObjConGradient)
     factor      K assembled and factored on the device; 0 = ok, k > 0 = non-positive pivot
                 in constraint k - 1, < 0 = bad arguments.  Dinv is kept by reference.
     apply3/4    yw = K^-1 (bw - A D^-1 bx), yx = D^-1 (bx + A^T yw)   (bw = 0 for apply3)
     mult_add, mult_transpose_add
                 out += alpha A px, out += alpha A^T pzw: ParOptSparseProblem's
                 addSparseJacobian / addSparseJacobianTranspose (ParOptProblem.cpp:756-816) */
typedef struct pcu_sparsemat pcu_sparsemat;
pcu_sparsemat *pcu_sparsemat_create(pcu_ctx *ctx, int nvars, int nwcon, const int *rowp,
                                    const int *cols, int ordering);
void pcu_sparsemat_destroy(pcu_sparsemat *mat);
int pcu_sparsemat_set_data(pcu_sparsemat *mat, const double *data);
double *pcu_sparsemat_data_device_ptr(pcu_sparsemat *mat);
int pcu_sparsemat_factor(pcu_sparsemat *mat, pcu_vec *x, pcu_vec *Dinv, pcu_vec *Cdiag);
int pcu_sparsemat_apply3(pcu_sparsemat *mat, pcu_vec *bx, pcu_vec *yx, pcu_vec *yw);
int pcu_sparsemat_apply4(pcu_sparsemat *mat, pcu_vec *bx, pcu_vec *bw, pcu_vec *yx,
                         pcu_vec *yw);
int pcu_sparsemat_mult_add(pcu_sparsemat *mat, double alpha, pcu_vec *px, pcu_vec *out);
int pcu_sparsemat_mult_transpose_add(pcu_sparsemat *mat, double alpha, pcu_vec *pzw,
                                     pcu_vec *out);
/* nnz of the lower triangles of K and of L, levels of the elimination tree, kernel
   launches of one factorisation (getFactorInfo, ParOptSparseMat.cpp:430-451)            */
int pcu_sparsemat_info(pcu_sparsemat *mat, int *nnzK, int *nnzL, int *nlevels,
                       int *nlaunches);
/* The symbolic factorisation as host arrays (sizes from pcu_sparsemat_info: perm nwcon,
   Lp nwcon + 1, Li nnzL, Rp nwcon + 1, Rk / Rpos nnzL - nwcon, kpos / ka / kb nnzK,
   level_ptr nlevels + 1, level_cols nwcon); NULL outputs are skipped.                   */
int pcu_sparsemat_symbolic(pcu_sparsemat *mat, int *perm, int *Lp, int *Li, int *Rp, int *Rk,
                           int *Rpos, int *kpos, int *ka, int *kb, int *level_ptr,
                           int *level_cols);

/* ---- ParOptCompactQuasiNewton (ParOptLBFGS / ParOptLSR1) as a stand-alone object
   (ParOptQuasiNewton.h:32-213): what ParOptInteriorPoint::setQuasiNewton or the
   trust-region front end is handed.  qn_type "bfgs" | "sr1".
     update      0 normal, 1 damped, 2 skipped in *update_type (QN.cpp:162-334, 636-747)
     mult        y = B x            (QN.cpp:390-418, 760-778)
     mult_add    y += alpha B x     (QN.cpp:432-459, 792-809)
     compact     returns q; b0, d0[q], M[q*q] column-major, Z[q] borrowed vectors
                 (QN.cpp:471-487, 821-837); any output may be NULL
     set_option  "qn_update_type" = skip_negative_curvature | damped_update,
                 "qn_diag_type" = yty_over_yts | yts_over_sts                     */
typedef struct pcu_qn pcu_qn;
pcu_qn *pcu_qn_create(pcu_ctx *ctx, int nvars, const char *qn_type, int subspace);
void pcu_qn_destroy(pcu_qn *qn);
int pcu_qn_set_option(pcu_qn *qn, const char *name, const char *value);
int pcu_qn_reset(pcu_qn *qn);
int pcu_qn_max_size(pcu_qn *qn);
int pcu_qn_update(pcu_qn *qn, pcu_vec *s, pcu_vec *y, int *update_type);
int pcu_qn_mult(pcu_qn *qn, pcu_vec *x, pcu_vec *y);
int pcu_qn_mult_add(pcu_qn *qn, double alpha, pcu_vec *x, pcu_vec *y);
int pcu_qn_compact(pcu_qn *qn, double *b0, double *d0, double *M, pcu_vec **Z);
/* ParOptInteriorPoint::setQuasiNewton (IP.cpp:1193): the optimizer uses (and, with
   use_quasi_newton_update, updates) the caller's object; NULL restores its own.  */
int pcu_ip_set_quasi_newton(pcu_ip *ip, pcu_qn *qn);

/* Host-array callbacks: the shape of a ParOptProblem whose callbacks work on
   ParOptVec::getArray pointers (ParOptProblem.h:143-172, ParOpt.pyx:520-640).
   The library owns page-locked host mirrors of x, g and the ncon constraint
   gradients (the arrays the callbacks see), copies the iterate device->host
   before a callback and the gradients host->device after it.  The copy of x is
   skipped when the optimizer knows the point is bit-identical to the one of the
   previous callback (accepted line-search trial, IP.cpp:4169-4215).            */
typedef struct pcu_host_callbacks {
  void *user;
  int (*get_vars_and_bounds)(void *user, int n, double *x, double *lb, double *ub);
  int (*eval_obj_con)(void *user, int n, const double *x, double *fobj,
                      double *cons);
  int (*eval_obj_con_gradient)(void *user, int n, const double *x, double *g,
                               double **Ac);
  /* Optional, as in pcu_problem_callbacks; writeOutput sees the iterate in the
     pinned host mirror (one device->host copy per call).                        */
  int (*write_output)(void *user, int iter, int n, const double *x);
  /* Optional, as in pcu_problem_callbacks: hvec = H(x, z, zw) px on host arrays
     (z: ncon values, zw: nw local sparse multipliers).                          */
  int (*eval_hvec_product)(void *user, int n, const double *x, const double *z, int nw,
                           const double *zw, const double *px, double *hvec);
} pcu_host_callbacks;
pcu_problem *pcu_problem_create_host(pcu_ctx *ctx, int nvars, int ncon,
                                     int ninequality, int nwinequality,
                                     int use_lower, int use_upper,
                                     const pcu_weighting *weighting,
                                     const pcu_host_callbacks *callbacks);
/* Bytes moved over PCIe by a host-array problem since its creation. */
int pcu_problem_transfer_bytes(pcu_problem *prob, int64_t *h2d, int64_t *d2h);
/* Wall-clock milliseconds a host-array problem spent copying the iterate to the
   host, inside the user callbacks, and (only with PCU_HOST_TIMING set, which
   synchronises after the uploads) copying the gradients to the device.        */
int pcu_problem_host_times(pcu_problem *prob, double *d2h_ms, double *user_ms,
                           double *h2d_ms);

/* ParOptProblem::evalHessianDiag: h = the diagonal of the Hessian of the Lagrangian at
   (x, z, zw), for the option use_diag_hessian, which uses diag(h) + qn_sigma in place of
   the quasi-Newton approximation.  The optimizer calls it once after every gradient
   evaluation, with the multipliers of that point (z: ncon host values); a non-zero return
   counts as a failed gradient evaluation.  The first form registers it on a problem of
   pcu_problem_create (pcu_vec handles, device memory), the second on one of
   pcu_problem_create_host (host arrays: x in the problem's mirror, zw copied to the host,
   h copied to the device after the call).  NULL unregisters; 1 for another kind of
   problem.  Built-in sepquad problems have the exact diagonal already.          */
int pcu_problem_set_hessian_diag(pcu_problem *prob, void *user,
                                 int (*eval_hessian_diag)(void *user, pcu_vec *x,
                                                          const double *z, pcu_vec *zw,
                                                          pcu_vec *h));
int pcu_problem_set_hessian_diag_host(pcu_problem *prob, void *user,
                                      int (*eval_hessian_diag)(void *user, int n,
                                                               const double *x,
                                                               const double *z, int nw,
                                                               const double *zw,
                                                               double *h));

/* MPI_Allreduce(MPI_SUM) stand-in for user callbacks that reduce their own
   partial sums (e.g. examples/rosenbrock/rosenbrock.cpp:100-117): `vals` are
   host doubles, summed over the ranks of the context in place.               */
int pcu_ctx_allreduce_sum(pcu_ctx *ctx, double *vals, int n);

/* Built-in GPU-resident synthetic problems (DESIGN.md "Synthetic problems");
   they implement the same three callbacks with CUDA kernels.
   Parameters of the separable / Householder convex QP family:                 */
typedef struct pcu_sepquad_params {
  int64_t ntotal;   /* GLOBAL number of design variables                       */
  int ncon;         /* dense constraints                                       */
  int nw;           /* variables per weighting block (0: none)                 */
  uint64_t seed;
  double lam_min, lam_max;
  double b_lo, b_w;
  double a_lo, a_w;
  double beta_c, beta_n, beta_u;
  double x0_lo[2], x0_w[2];
  double lb[2], ub[2];
  int householder;
} pcu_sepquad_params;
pcu_problem *pcu_problem_create_sepquad(pcu_ctx *ctx,
                                        const pcu_sepquad_params *params);
/* The same workload as a HOST problem: C++ callbacks over host arrays, threaded
   over `nthreads` host cores (<= 0: all), registered through
   pcu_problem_create_host -- what the end-to-end benchmark drives.  `user_out`
   receives the callback state; free it with pcu_problem_sepquad_host_free after
   pcu_problem_destroy.                                                        */
pcu_problem *pcu_problem_create_sepquad_host(pcu_ctx *ctx,
                                             const pcu_sepquad_params *params,
                                             int nthreads, void **user_out);
void pcu_problem_sepquad_host_free(void *user);
/* examples/rosenbrock/rosenbrock.cpp:9-199 (single rank). */
pcu_problem *pcu_problem_create_rosenbrock(pcu_ctx *ctx, int nvars, int nwcon,
                                           int nwstart, int nw, int nwskip);
int pcu_problem_sizes(pcu_problem *prob, int *nvars, int *ncon, int *nwcon);
/* Seconds spent inside the problem callbacks (device time, user code). */
double pcu_problem_callback_ms(pcu_problem *prob);

/* --------------------------------------------------- interior-point optimizer
   ParOptInteriorPoint public API (ParOptInteriorPoint.h:128-217).             */
pcu_ip *pcu_ip_create(pcu_problem *prob);                  /* IP.cpp:182       */
void pcu_ip_destroy(pcu_ip *ip);
/* ParOptOptions::setOption (ParOptOptions.h:35-37); names, defaults and ranges
   as registered by addDefaultOptions (IP.cpp:536-727).  Unknown name -> 1.
   use_diag_hessian (0/1) takes the problem's evalHessianDiag as the Hessian; no
   quasi-Newton object is built and qn_type is ignored.  It runs with the monotone
   barrier, iterative_refinement_steps = 1 and 1..32 dense constraints; begin /
   optimize refuse it (non-zero, one "ParOpt error:" line) without the callback, with
   use_hvec_product, sequential_linear_method or a pcu_ip_set_quasi_newton object. */
int pcu_ip_set_option_float(pcu_ip *ip, const char *name, double value);
int pcu_ip_set_option_int(pcu_ip *ip, const char *name, int value);
int pcu_ip_set_option_str(pcu_ip *ip, const char *name, const char *value);
/* optimize (IP.cpp:4399).  Returns 0 on completion. */
int pcu_ip_optimize(pcu_ip *ip);
/* The same major loop, resumable: begin = everything before the loop
   (IP.cpp:4399-4606), iterate = up to `max_iters` passes of the loop body
   (IP.cpp:4607-5329); *converged is set when the convergence test fires.       */
int pcu_ip_begin(pcu_ip *ip);
int pcu_ip_iterate(pcu_ip *ip, int max_iters, int *converged);
/* resetDesignAndBounds (IP.cpp:1249): asks the problem for x, lb, ub again.     */
int pcu_ip_reset_design_and_bounds(pcu_ip *ip);
/* setPenaltyGamma(double) (IP.cpp:1128) and setPenaltyGamma(const double*)
   (IP.cpp:1160; ncon values, negative entries keep the current value; the sparse
   penalties keep the scalar).                                                  */
int pcu_ip_set_penalty_gamma(pcu_ip *ip, double gamma);
int pcu_ip_set_penalty_gamma_array(pcu_ip *ip, const double *gamma);
int pcu_ip_get_penalty_gamma(pcu_ip *ip, double *gamma_t);   /* penalty_gamma_t, IP.h:431 */
/* resetProblemInstance (IP.cpp:745): a problem of identical sizes, inequality
   counts and weighting descriptor replaces the current one; 1 = incompatible.   */
int pcu_ip_reset_problem(pcu_ip *ip, pcu_problem *prob);
/* resetQuasiNewtonHessian (IP.cpp:1241).                                        */
int pcu_ip_reset_quasi_newton(pcu_ip *ip);
/* writeSolutionFile / readSolutionFile (IP.cpp:883-975, 986-1104): the reference's
   binary checkpoint, byte for byte -- int[3] {global nvars, global nwcon, ncon},
   barrier, s, t, z, zs, zt (ncon doubles each), then x, zl, zu (global nvars each) and
   zw, sw (global nwcon each) in rank order; every rank writes / reads its own slice.
   The option "ip_checkpoint_file" makes optimize() write it at every
   write_output_frequency-th iteration (IP.cpp:4621-4629).  1 on failure (a size
   mismatch prints the reference's message).                                      */
int pcu_ip_write_solution(pcu_ip *ip, const char *filename);
int pcu_ip_read_solution(pcu_ip *ip, const char *filename);
/* getOptimizedPoint / getOptimizedSlacks (IP.h:156-163): device vectors owned
   by the optimizer plus host copies of the dense parts.                       */
int pcu_ip_get_point(pcu_ip *ip, pcu_vec **x, pcu_vec **zw, pcu_vec **zl,
                     pcu_vec **zu, pcu_vec **sw, pcu_vec **tw);
int pcu_ip_get_dense(pcu_ip *ip, double *z, double *s, double *t, double *zs,
                     double *zt, double *c);
double pcu_ip_barrier_param(pcu_ip *ip);       /* getBarrierParameter IP.h:177 */
int pcu_ip_complementarity(pcu_ip *ip, double *comp); /* getComplementarity    */
int pcu_ip_counters(pcu_ip *ip, int *niter, int *neval, int *ngeval);
/* 0 none, 1 "converged to requested tolerance", 2 relative function test,
   3 "could not be improved" (the three messages at IP.cpp:4815-4830).         */
int pcu_ip_status(pcu_ip *ip);

/* -------------------------------------------------- trust-region front end
   ParOptTrustRegion with the SL1QP penalty method and the adaptive penalty update
   (src/ParOptTrustRegion.cpp:1454-1690) over ParOptQuadraticSubproblem /
   ParOptInfeasSubproblem model problems that live on the device (TR.cpp:27-660) --
   what ParOptOptimizer runs for algorithm = "tr" (src/ParOptOptimizer.cpp:102-175).
   Options: the tr_* names of ParOptTrustRegion::addDefaultOptions (TR.cpp:739-845),
   the qn_* names, and every interior-point option (forwarded to the subproblem
   optimizer).  Not built: tr_accept_step_strategy = filter_method, tr_use_soc.     */
typedef struct pcu_tr pcu_tr;
pcu_tr *pcu_tr_create(pcu_problem *prob);
void pcu_tr_destroy(pcu_tr *tr);
int pcu_tr_set_option_float(pcu_tr *tr, const char *name, double value);
int pcu_tr_set_option_int(pcu_tr *tr, const char *name, int value);
int pcu_tr_set_option_str(pcu_tr *tr, const char *name, const char *value);
int pcu_tr_optimize(pcu_tr *tr);                 /* TR.cpp:2367 optimize            */
int pcu_tr_status(pcu_tr *tr);                   /* 1: converged (TR.cpp:1603-1608) */
/* One record per trust-region iteration, the columns of the reference's log row
   (TR.cpp:1433-1445) at full precision plus checksums of the centre x_k:
   iter fobj infeas l1 linfty |x-xk| tr rho model_red zav zmax gav gmax
   subproblem_iters adaptive_iters accepted xsum xnorm xmaxabs (19 doubles).        */
int pcu_tr_history_len(pcu_tr *tr);
int pcu_tr_history_get(pcu_tr *tr, int k, double *out19);
const char *pcu_tr_history_info(pcu_tr *tr, int k);
pcu_vec *pcu_tr_point(pcu_tr *tr);               /* getOptimizedPoint TR.cpp:888    */
pcu_ip *pcu_tr_interior_point(pcu_tr *tr);       /* the subproblem optimizer        */
int pcu_tr_penalty_gamma(pcu_tr *tr, double *gamma);   /* getPenaltyGamma TR.cpp:1076 */

/* Per-iteration history at the point of the reference's writeOutput hook
   (IP.cpp:4620-4631): one record per major iteration, PCU_HIST_FIELDS doubles
   followed by 6*ncon doubles (c, z, s, t, zs, zt).  Field order:
   iter fobj mu rho comp max_prime max_dual max_infeas res_norm neval ngeval
   alpha pnorm2 qn_b0 qn_size xsum xnorm zlsum zusum zwsum swsum twsum gmax
   alpha_x alpha_z nhvec                                                      */
#define PCU_HIST_FIELDS 26
int pcu_ip_history_len(pcu_ip *ip);
int pcu_ip_history_get(pcu_ip *ip, int k, double *out, int out_len);
/* The `info` tag string of the log row printed at iteration k (IP.cpp:5272).  */
const char *pcu_ip_history_info(pcu_ip *ip, int k);
/* Device milliseconds of each completed major iteration and the share spent in
   problem callbacks and in the KKT solve (setUpKKTDiagSystem + setUpKKTSystem
   + first computeKKTStep).                                                    */
int pcu_ip_iter_times(pcu_ip *ip, int k, double *total_ms, double *callback_ms,
                      double *kkt_ms);

/* ---------------------------------------------- hot-path functions, one by one
   (kernel-level parity tests drive these; each acts on the optimizer's own
   state exactly as the private method of the same name does).  `which` selects
   a ParOptVars bundle: 0 variables, 1 residual, 2 update, 3 refine
   (ParOptInteriorPoint.h:413-416).                                            */
enum { PCU_VARS = 0, PCU_RESIDUAL = 1, PCU_UPDATE = 2, PCU_REFINE = 3 };
/* component ids for pcu_ip_vars_vec */
enum { PCU_X = 0, PCU_ZL, PCU_ZU, PCU_ZW, PCU_SW, PCU_TW, PCU_ZSW, PCU_ZTW };
pcu_vec *pcu_ip_vars_vec(pcu_ip *ip, int which, int component);
/* dense parts: 5*ncon doubles in the order z, s, t, zs, zt */
int pcu_ip_vars_dense_get(pcu_ip *ip, int which, double *out5c);
int pcu_ip_vars_dense_set(pcu_ip *ip, int which, const double *in5c);
/* other state vectors: 0 lb, 1 ub, 2 g, 3 Dinv, 4 Cw(factor), 100+j Ac[j]      */
pcu_vec *pcu_ip_state_vec(pcu_ip *ip, int id);
int pcu_ip_set_obj_con(pcu_ip *ip, double fobj, const double *c);
int pcu_ip_set_barrier(pcu_ip *ip, double mu, double rho);
/* Loads the quasi-Newton memory from host arrays (S, Y: msub vectors of n) by
   replaying ParOptLBFGS/LSR1::update (QN.cpp:162 / :636) on the device.       */
int pcu_ip_qn_update(pcu_ip *ip, pcu_vec *s, pcu_vec *y, int *update_type);
int pcu_ip_qn_reset(pcu_ip *ip);                                /* QN.cpp:132  */
int pcu_ip_qn_mult(pcu_ip *ip, pcu_vec *x, pcu_vec *y);         /* QN.cpp:390  */
int pcu_ip_qn_compact(pcu_ip *ip, double *b0, int *size, double *d0,
                      double *M);                               /* QN.cpp:471  */

int pcu_ip_kkt_res(pcu_ip *ip, int vars, double mu, int res);   /* IP.cpp:1337 */
int pcu_ip_res_norm(pcu_ip *ip, double *max_prime, double *max_dual,
                    double *max_infeas, double *res_norm);       /* IP.cpp:1588 */
int pcu_ip_comp(pcu_ip *ip, double *comp);                       /* IP.cpp:2742 */
int pcu_ip_setup_kkt_diag(pcu_ip *ip, int use_qn);               /* IP.cpp:1832 */
int pcu_ip_setup_kkt(pcu_ip *ip, int use_qn);                    /* IP.cpp:2634 */
int pcu_ip_kkt_step(pcu_ip *ip, int res, int step, int use_qn);  /* IP.cpp:2700 */
int pcu_ip_add_kkt_res_step(pcu_ip *ip, int step, int res);      /* IP.cpp:1451 */
/* The KKT solve of the default iteration (one refinement step, done in the column
   space of [A|Z]) at the current point and barrier, right-hand side from the
   variables, dense algebra on the device (on_device = 1) or on the host; needs
   1 <= ncon + quasi-Newton width <= 32.  res receives the dense residual only. */
int pcu_ip_kkt_solve(pcu_ip *ip, int res, int step, int on_device); /* IP.cpp:4971 */
int pcu_ip_max_step(pcu_ip *ip, double tau, int step, double *max_x,
                    double *max_z);                              /* IP.cpp:2942 */
int pcu_ip_comp_step(pcu_ip *ip, double alpha_x, double alpha_z, int step,
                     double *comp);                              /* IP.cpp:2825 */
int pcu_ip_merit_init_deriv(pcu_ip *ip, double max_x, double *merit,
                            double *pmerit);                     /* IP.cpp:3652 */
/* Gram blocks of the last setup: G (ncon x ncon, col-major, before LU) and
   Ce (q x q, col-major, before LU) -- IP.cpp:1932-1961 and 2646-2661.         */
int pcu_ip_get_gram(pcu_ip *ip, double *G, double *Ce, int *q);
/* Work partition of the wide Gram kernel (more than 40 columns: the A^T D^-1 A / Z^T D^-1 Z
   contraction of setUpKKTDiagSystem / setUpKKTSystem, IP.cpp:1932-1961, 2646-2661, on the
   FP64 tensor cores) for m columns, as host arrays -- inspection and CPU tests, no device
   call: nt tile rows of 8 columns, n2u common two-pair segments per consumer warp, side = 1
   when the last column is taken as a side column; ti / tj / np [warps][slots]: tile row,
   first tile column and number of tile pairs (0 = empty slot) of every segment.  NULL
   tables are skipped; returns non-zero when the wide kernel does not take this width.   */
int pcu_gram_wide_plan(int m, int *nt, int *n2u, int *side, int *warps, int *slots,
                       unsigned char *ti, unsigned char *tj, unsigned char *np);

#ifdef __cplusplus
}
#endif

#endif /* PAROPT_B200_H */
