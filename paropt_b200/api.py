"""Host-side mirror of the reference's Python surface for the interior-point path
(paropt/ParOpt.pyx: PVec :914, Problem :787, InteriorPoint :1189), bound to the
C ABI in include/paropt_b200.h through ctypes.

Everything numerical runs in libparopt_b200.so on the GPU; this module only
marshals arguments.  There is no CPU fallback: constructing a Context without a
CUDA device raises RuntimeError.
"""
import ctypes as C

import numpy as np

from . import _lib

HIST_FIELDS = ("iter", "fobj", "mu", "rho", "comp", "max_prime", "max_dual",
               "max_infeas", "res_norm", "neval", "ngeval", "alpha", "pnorm2",
               "qn_b0", "qn_size", "xsum", "xnorm", "zlsum", "zusum", "zwsum",
               "swsum", "twsum", "gmax", "alpha_x", "alpha_z", "nhvec")
STATUS = {0: None, 1: "tolerance", 2: "rel_function", 3: "no_improvement"}


def _check(rc, what):
    if rc != 0:
        raise RuntimeError("paropt_b200: %s failed (code %d)" % (what, rc))


class Context:
    """One per process / GPU (replaces the MPI communicator)."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        self.h = self.lib.pcu_ctx_create(int(device))
        if not self.h:
            raise RuntimeError(
                "paropt_b200: could not create a CUDA context on device %d; the "
                "interior-point core has no CPU fallback" % device)
        self.device = int(device)
        self.rank, self.size = 0, 1
        self._stream = None

    @property
    def stream(self):
        """The context's CUDA stream (pcu_ctx_stream) as a torch.cuda.ExternalStream:
        torch work enqueued there is ordered with the library's kernels."""
        if self._stream is None:
            import torch
            self._stream = torch.cuda.ExternalStream(
                int(self.lib.pcu_ctx_stream(self.h)), device=torch.device("cuda", self.device))
        return self._stream

    def allreduce_sum(self, values):
        """Sum of `values` (host numbers, or a tensor) over the ranks of the context
        (pcu_ctx_allreduce_sum; MPI_Allreduce(MPI_SUM) in the reference's examples),
        as a float64 numpy array."""
        if hasattr(values, "detach"):
            values = values.detach().cpu().numpy()
        out = np.array(values, dtype=np.float64).ravel()
        if out.size:
            _check(self.lib.pcu_ctx_allreduce_sum(self.h, out.ctypes.data_as(_lib.c_double_p),
                                                  out.size), "allreduce_sum")
        return out

    def init_distributed(self):
        """Bootstraps the NCCL communicator of this context from an initialised
        torch.distributed process group (one process per GPU)."""
        import torch
        import torch.distributed as dist

        rank, world = dist.get_rank(), dist.get_world_size()
        buf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = C.create_string_buffer(128)
            _check(self.lib.pcu_nccl_unique_id(raw), "ncclGetUniqueId")
            buf = torch.tensor(list(raw.raw), dtype=torch.uint8)
        if dist.get_backend() == "nccl":
            dev = torch.device("cuda", torch.cuda.current_device())
            tmp = buf.to(dev)
            dist.broadcast(tmp, 0)
            buf = tmp.cpu()
        else:
            dist.broadcast(buf, 0)
        raw = bytes(buf.tolist())
        _check(self.lib.pcu_ctx_init_comm(self.h, raw, rank, world), "ncclCommInitRank")
        self.rank, self.size = rank, world

    def sync(self):
        _check(self.lib.pcu_ctx_sync(self.h), "sync")

    def kernel_launches(self):
        return int(self.lib.pcu_ctx_kernel_launches(self.h))

    def set_param(self, name, value):
        """Launch tuning knob (include/paropt_b200.h: pcu_ctx_set_param)."""
        _check(self.lib.pcu_ctx_set_param(self.h, name.encode(), int(value)), "set_param " + name)

    def profile(self, enable):
        _check(self.lib.pcu_ctx_profile(self.h, int(enable)), "profile")

    def profile_totals(self):
        """{kernel name: (total ms, launches)} accumulated while profiling."""
        out = {}
        n = int(self.lib.pcu_ctx_profile_count(self.h))
        name = C.create_string_buffer(256)
        ms, cnt = C.c_double(), C.c_int64()
        for i in range(n):
            if self.lib.pcu_ctx_profile_get(self.h, i, name, 256, C.byref(ms),
                                            C.byref(cnt)) == 0:
                out[name.value.decode()] = (ms.value, int(cnt.value))
        return out

    def timer_start(self):
        _check(self.lib.pcu_ctx_timer_start(self.h), "timer_start")

    def timer_stop(self):
        ms = C.c_double()
        _check(self.lib.pcu_ctx_timer_stop(self.h, C.byref(ms)), "timer_stop")
        return ms.value

    def close(self):
        if self.h:
            self.lib.pcu_ctx_destroy(self.h)
            self.h = None


class PVec:
    """ParOptVec / PVec (ParOptVec.h:53-70, ParOpt.pyx:914) in device memory."""

    def __init__(self, ctx, n=None, handle=None):
        self.ctx = ctx
        self.lib = ctx.lib
        self.owns = handle is None
        self.h = handle if handle is not None else self.lib.pcu_vec_create(ctx.h, int(n))
        if not self.h:
            raise RuntimeError("paropt_b200: vector allocation failed")

    def __len__(self):
        return int(self.lib.pcu_vec_size(self.h))

    def set(self, alpha):
        _check(self.lib.pcu_vec_set(self.h, float(alpha)), "set")

    def zeroEntries(self):
        _check(self.lib.pcu_vec_zero(self.h), "zeroEntries")

    def copyValues(self, other):
        _check(self.lib.pcu_vec_copy(self.h, other.h), "copyValues")

    def norm(self):
        out = C.c_double()
        _check(self.lib.pcu_vec_norm(self.h, C.byref(out)), "norm")
        return out.value

    def maxabs(self):
        out = C.c_double()
        _check(self.lib.pcu_vec_maxabs(self.h, C.byref(out)), "maxabs")
        return out.value

    def l1norm(self):
        out = C.c_double()
        _check(self.lib.pcu_vec_l1norm(self.h, C.byref(out)), "l1norm")
        return out.value

    def dot(self, other):
        out = C.c_double()
        _check(self.lib.pcu_vec_dot(self.h, other.h, C.byref(out)), "dot")
        return out.value

    def mdot(self, vecs):
        k = len(vecs)
        arr = (C.c_void_p * k)(*[v.h for v in vecs])
        out = np.zeros(k)
        _check(self.lib.pcu_vec_mdot(self.h, arr, k, out.ctypes.data_as(_lib.c_double_p)), "mdot")
        return out

    def scale(self, alpha):
        _check(self.lib.pcu_vec_scale(self.h, float(alpha)), "scale")

    def axpy(self, alpha, x):
        _check(self.lib.pcu_vec_axpy(self.h, float(alpha), x.h), "axpy")

    def device_ptr(self):
        return int(self.lib.pcu_vec_device_ptr(self.h) or 0)

    def host_array(self):
        """numpy view of a managed vector (Context.set_param("managed_vectors", 1)):
        ParOptVec::getArray for host loops; reads and writes go to the vector itself."""
        ptr = self.lib.pcu_vec_host_ptr(self.h)
        if not ptr:
            raise RuntimeError("paropt_b200: not a managed vector")
        n = len(self)
        return np.ctypeslib.as_array(C.cast(ptr, _lib.c_double_p), shape=(n,)) if n else np.empty(0)

    # Zero-copy device view (torch.as_tensor(v, device="cuda"), cupy.asarray(v)):
    # the fast path SURVEY.md section 8f-2 asks for instead of PVec's per-element
    # host indexing (ParOpt.pyx:1082-1159).
    @property
    def __cuda_array_interface__(self):
        return {"shape": (len(self),), "typestr": "<f8",
                "data": (self.device_ptr(), False), "version": 3, "strides": None}

    # Host-side element access with the reference's semantics (ParOpt.pyx:1082-
    # 1159: integers and slices); every access is a device<->host copy of the
    # touched range's vector, meant for set-up and inspection, not for loops.
    def __array__(self, dtype=None, copy=None):
        a = self.to_numpy()
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, key):
        return self.to_numpy()[key]

    def __setitem__(self, key, value):
        a = self.to_numpy()
        a[key] = value
        self.from_numpy(a)

    def to_numpy(self):
        out = np.empty(len(self))
        if len(self):
            _check(self.lib.pcu_vec_to_host(self.h, out.ctypes.data, len(self)), "to_host")
        return out

    def from_numpy(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float64)
        if arr.size != len(self):
            raise ValueError("size mismatch")
        if arr.size:
            _check(self.lib.pcu_vec_from_host(self.h, arr.ctypes.data, arr.size), "from_host")

    def free(self):
        if self.owns and self.h:
            self.lib.pcu_vec_destroy(self.h)
            self.h = None


class QuasiDefBlockMat:
    """ParOptQuasiDefBlockMat, nwblock = 1 (ParOptSparseMat.h:64-104) for the
    weighting rows of a `weighting` dict (nwcon, wstart, nw, wstride, coef0,
    coef_rest, wconst)."""

    def __init__(self, ctx, nvars, weighting=None, blocks=None):
        """weighting: nwblock = 1 rows (pcu_weighting).  blocks: the block form with
        nwblock = nb > 1 -- dict(nblocks, wstart, nw, wstride, coef=[nb][nw] array)
        (pcu_block_weighting, ParOptSparseMat.cpp:72-111, 196-224)."""
        self.ctx, self.lib = ctx, ctx.lib
        if blocks is not None:
            coef = np.ascontiguousarray(blocks["coef"], dtype=np.float64)
            nb, nw = coef.shape
            b = _lib.BlockWeighting()
            b.nblocks, b.wstart, b.nw = int(blocks["nblocks"]), int(blocks.get("wstart", 0)), nw
            b.wstride, b.nb = int(blocks.get("wstride", nw)), nb
            b.coef = coef.ctypes.data_as(_lib.c_double_p)
            b.wconst = None
            self.nvars, self.nwcon = int(nvars), b.nblocks * nb
            self.h = self.lib.pcu_blockmat_create_blocks(ctx.h, int(nvars), C.byref(b))
            if not self.h:
                raise RuntimeError("paropt_b200: pcu_blockmat_create_blocks failed")
            return
        w = _lib.Weighting()
        for k, v in (weighting or {}).items():
            setattr(w, k, v)
        self.nvars, self.nwcon = int(nvars), int(w.nwcon)
        self.h = self.lib.pcu_blockmat_create(ctx.h, int(nvars), C.byref(w))
        if not self.h:
            raise RuntimeError("paropt_b200: pcu_blockmat_create failed")

    def factor(self, x, Dinv, Cdiag):
        """0 = ok, k > 0: zero pivot in row k - 1 (ParOptSparseMat.cpp:41-115)."""
        rc = int(self.lib.pcu_blockmat_factor(self.h, x.h if x is not None else None,
                                              Dinv.h, Cdiag.h))
        if rc < 0:
            raise RuntimeError("paropt_b200: pcu_blockmat_factor: bad arguments")
        return rc

    def apply(self, bx, *rest):
        """apply(bx, yx, yw) / apply(bx, bw, yx, yw) (ParOptSparseMat.cpp:122-190)."""
        if len(rest) == 2:
            _check(self.lib.pcu_blockmat_apply3(self.h, bx.h, rest[0].h, rest[1].h), "apply")
        else:
            bw, yx, yw = rest
            _check(self.lib.pcu_blockmat_apply4(self.h, bx.h, bw.h, yx.h, yw.h), "apply")

    def free(self):
        if self.h:
            self.lib.pcu_blockmat_destroy(self.h)
            self.h = None


class QuasiDefSparseMat:
    """ParOptQuasiDefSparseMat (ParOptSparseMat.cpp:231-451) for a CSR constraint Jacobian
    (rowp, cols; ParOptSparseProblem.setSparseJacobianData): K = C + A D^-1 A^T assembled
    and factored on the device (pcu_sparsemat).  ordering: "minimum_degree" | "natural"."""

    def __init__(self, ctx, nvars, nwcon, rowp, cols, ordering="minimum_degree"):
        self.ctx, self.lib = ctx, ctx.lib
        self.nvars, self.nwcon = int(nvars), int(nwcon)
        rowp = np.ascontiguousarray(rowp, dtype=np.int32)
        cols = np.ascontiguousarray(cols if len(cols) else [0], dtype=np.int32)
        self.nnz = int(rowp[-1])
        self.h = self.lib.pcu_sparsemat_create(
            ctx.h, self.nvars, self.nwcon, rowp.ctypes.data_as(_lib.c_int_p),
            cols.ctypes.data_as(_lib.c_int_p), 1 if ordering == "minimum_degree" else 0)
        if not self.h:
            raise RuntimeError("paropt_b200: pcu_sparsemat_create failed")

    def set_data(self, data):
        data = np.ascontiguousarray(data, dtype=np.float64)
        if data.size != self.nnz:
            raise ValueError("expected %d Jacobian values" % self.nnz)
        if self.nnz:
            _check(self.lib.pcu_sparsemat_set_data(self.h, data.ctypes.data_as(_lib.c_double_p)),
                   "set_data")

    def factor(self, x, Dinv, Cdiag):
        """0 = ok, k > 0: non-positive pivot in constraint k - 1."""
        rc = int(self.lib.pcu_sparsemat_factor(self.h, x.h if x is not None else None,
                                               Dinv.h, Cdiag.h))
        if rc < 0:
            raise RuntimeError("paropt_b200: pcu_sparsemat_factor: bad arguments")
        return rc

    def apply(self, bx, *rest):
        if len(rest) == 2:
            _check(self.lib.pcu_sparsemat_apply3(self.h, bx.h, rest[0].h, rest[1].h), "apply")
        else:
            bw, yx, yw = rest
            _check(self.lib.pcu_sparsemat_apply4(self.h, bx.h, bw.h, yx.h, yw.h), "apply")

    def mult_add(self, alpha, px, out):
        _check(self.lib.pcu_sparsemat_mult_add(self.h, float(alpha), px.h, out.h), "mult_add")

    def mult_transpose_add(self, alpha, pzw, out):
        _check(self.lib.pcu_sparsemat_mult_transpose_add(self.h, float(alpha), pzw.h, out.h),
               "mult_transpose_add")

    def info(self):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self.lib.pcu_sparsemat_info(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
        return dict(nnzK=a.value, nnzL=b.value, levels=c.value, launches=d.value)

    def free(self):
        if self.h:
            self.lib.pcu_sparsemat_destroy(self.h)
            self.h = None


class QuasiNewton:
    """ParOptLBFGS / ParOptLSR1 (ParOptQuasiNewton.h:76-213; ParOpt.pyx LBFGS/LSR1)."""

    def __init__(self, ctx, nvars, qn_type="bfgs", subspace=10):
        self.ctx, self.lib = ctx, ctx.lib
        self.h = self.lib.pcu_qn_create(ctx.h, int(nvars), qn_type.encode(), int(subspace))
        if not self.h:
            raise RuntimeError("paropt_b200: pcu_qn_create failed")

    def set_option(self, name, value):
        _check(self.lib.pcu_qn_set_option(self.h, name.encode(), str(value).encode()),
               "qn option " + name)

    def reset(self):
        _check(self.lib.pcu_qn_reset(self.h), "qn reset")

    def getMaxLimitedMemorySize(self):
        return int(self.lib.pcu_qn_max_size(self.h))

    def update(self, s, y):
        ut = C.c_int()
        _check(self.lib.pcu_qn_update(self.h, s.h, y.h, C.byref(ut)), "qn update")
        return ut.value

    def mult(self, x, y):
        _check(self.lib.pcu_qn_mult(self.h, x.h, y.h), "qn mult")

    def multAdd(self, alpha, x, y):
        _check(self.lib.pcu_qn_mult_add(self.h, float(alpha), x.h, y.h), "qn multAdd")

    def getCompactMat(self):
        """(b0, d0, M, Z): M is q x q (column-major in the library, returned as a
        numpy array with M[i, j] = entry (i, j)); Z is a list of borrowed PVec."""
        q = int(self.lib.pcu_qn_compact(self.h, None, None, None, None))
        b0 = C.c_double()
        d0 = np.zeros(max(q, 1))
        M = np.zeros(max(q * q, 1))
        Z = (C.c_void_p * max(q, 1))()
        self.lib.pcu_qn_compact(self.h, C.byref(b0), d0.ctypes.data_as(_lib.c_double_p),
                                M.ctypes.data_as(_lib.c_double_p), Z)
        Mm = M[:q * q].reshape(q, q).T.copy()
        return b0.value, d0[:q], Mm, [PVec(self.ctx, handle=Z[i]) for i in range(q)]

    def free(self):
        if self.h:
            self.lib.pcu_qn_destroy(self.h)
            self.h = None


def sepquad_params(**kw):
    p = _lib.SepQuadParams()
    defaults = dict(ntotal=1000, ncon=1, nw=0, seed=0, lam_min=1.0, lam_max=1e3,
                    b_lo=0.0, b_w=1.0, a_lo=0.0, a_w=1.0, beta_c=0.0, beta_n=0.0,
                    beta_u=1.0, x0_lo0=-2.0, x0_lo1=-2.0, x0_w0=1.0, x0_w1=1.0,
                    lb0=-5.0, lb1=-5.0, ub0=5.0, ub1=5.0, householder=0)
    for k in kw:
        if k not in defaults:
            raise ValueError("unknown sepquad parameter %s" % k)
    defaults.update(kw)
    d = defaults
    for name in ("ntotal", "ncon", "nw", "seed", "lam_min", "lam_max", "b_lo", "b_w",
                 "a_lo", "a_w", "beta_c", "beta_n", "beta_u", "householder"):
        setattr(p, name, d[name])
    p.x0_lo[0], p.x0_lo[1] = d["x0_lo0"], d["x0_lo1"]
    p.x0_w[0], p.x0_w[1] = d["x0_w0"], d["x0_w1"]
    p.lb[0], p.lb[1] = d["lb0"], d["lb1"]
    p.ub[0], p.ub[1] = d["ub0"], d["ub1"]
    return p


class Problem:
    """ParOpt.Problem (ParOpt.pyx:787-907): subclass and implement
    getVarsAndBounds(x, lb, ub), evalObjCon(x) -> (fail, fobj, con) and
    evalObjConGradient(x, g, A) -> fail on numpy arrays.  The arrays are views
    of page-locked host mirrors owned by the library (the reference's getArray
    contract, pcu_problem_create_host); each callback costs one device->host
    copy of the iterate (skipped when the point is the one the previous callback
    saw) and one host->device copy of the vectors it fills."""

    def __init__(self, ctx, nvars, ncon, ninequality=-1, nwinequality=-1,
                 use_lower=True, use_upper=True, weighting=None):
        self.ctx = ctx
        self.lib = ctx.lib
        self.nvars, self.ncon = int(nvars), int(ncon)
        w = _lib.Weighting()
        if weighting:
            for k, v in weighting.items():
                setattr(w, k, v)
        self._w = w
        self._cb = _lib.HostCallbacks()
        self._cb.user = None
        self._cb.get_vars_and_bounds = _lib.HOST_GET_VARS_CB(self._get_vars)
        self._cb.eval_obj_con = _lib.HOST_EVAL_OBJ_CB(self._eval_obj)
        self._cb.eval_obj_con_gradient = _lib.HOST_EVAL_GRAD_CB(self._eval_grad)
        # ParOptProblem::writeOutput (ParOptProblem.h:296): registered only when the
        # subclass defines it, so that nobody pays the device->host copy otherwise
        if hasattr(self, "writeOutput"):
            self._cb.write_output = _lib.HOST_WRITE_OUT_CB(self._write_output)
        # ParOptProblem::evalHvecProduct (ParOptProblem.h:188; ParOpt.pyx _evalhvecproduct):
        # evalHvecProduct(x, z, zw, px, hvec) -> fail, for the option use_hvec_product
        if hasattr(self, "evalHvecProduct"):
            self._cb.eval_hvec_product = _lib.HOST_HVEC_CB(self._eval_hvec)
        self._views = {}
        self.h = self.lib.pcu_problem_create_host(
            ctx.h, self.nvars, self.ncon, int(ninequality), int(nwinequality),
            int(use_lower), int(use_upper), C.byref(self._w), C.byref(self._cb))
        if not self.h:
            raise RuntimeError("paropt_b200: problem creation failed")
        # ParOptProblem::evalHessianDiag: evalHessianDiag(x, z, zw, hdiag) -> fail, for the
        # option use_diag_hessian
        if hasattr(self, "evalHessianDiag"):
            self._hdiag_cb = _lib.HOST_HDIAG_CB(self._eval_hdiag)
            _check(self.lib.pcu_problem_set_hessian_diag_host(self.h, None, self._hdiag_cb),
                   "set_hessian_diag_host")

    def _view(self, ptr, n):
        """numpy view of a library-owned host array (cached per address)."""
        addr = C.addressof(ptr.contents) if n > 0 else 0
        v = self._views.get(addr)
        if v is None or v.shape[0] != n:
            v = np.ctypeslib.as_array(ptr, shape=(n,)) if n > 0 else np.empty(0)
            self._views[addr] = v
        return v

    @property
    def h2d_bytes(self):
        a, b = C.c_int64(), C.c_int64()
        self.lib.pcu_problem_transfer_bytes(self.h, C.byref(a), C.byref(b))
        return a.value

    @property
    def d2h_bytes(self):
        a, b = C.c_int64(), C.c_int64()
        self.lib.pcu_problem_transfer_bytes(self.h, C.byref(a), C.byref(b))
        return b.value

    def _get_vars(self, user, n, x, lb, ub):
        try:
            self.getVarsAndBounds(self._view(x, n), self._view(lb, n), self._view(ub, n))
            return 0
        except Exception:  # mirrors ParOpt.pyx:528-531 (report, do not unwind C)
            import traceback
            traceback.print_exc()
            return 1

    def _eval_obj(self, user, n, x, fobj, cons):
        try:
            fail, f, con = self.evalObjCon(self._view(x, n))
            fobj[0] = float(f)
            for i in range(self.ncon):
                cons[i] = float(con[i])
            return int(fail)
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def _eval_hvec(self, user, n, x, z, nw, zw, px, hvec):
        try:
            zz = np.array([z[i] for i in range(self.ncon)])
            fail = self.evalHvecProduct(self._view(x, n), zz, self._view(zw, nw),
                                        self._view(px, n), self._view(hvec, n))
            return int(fail or 0)
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def _eval_hdiag(self, user, n, x, z, nw, zw, hdiag):
        try:
            zz = np.array([z[i] for i in range(self.ncon)])
            fail = self.evalHessianDiag(self._view(x, n), zz, self._view(zw, nw),
                                        self._view(hdiag, n))
            return int(fail or 0)
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def _write_output(self, user, it, n, x):
        try:
            self.writeOutput(int(it), self._view(x, n))
            return 0
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def _eval_grad(self, user, n, x, g, Ac):
        try:
            A = [self._view(Ac[i], n) for i in range(self.ncon)]
            fail = self.evalObjConGradient(self._view(x, n), self._view(g, n), A)
            return int(fail or 0)
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def free(self):
        if self.h:
            self._views.clear()
            self.lib.pcu_problem_destroy(self.h)
            self.h = None


class _DeviceArray:
    """A library-owned device range in the CUDA array interface (no stream key: the
    callbacks order the streams themselves)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False),
                                         "version": 3, "strides": None}


class TorchProblem:
    """ParOpt.Problem with callbacks on torch tensors in device memory
    (pcu_problem_create): subclass and implement

        getVarsAndBounds(x, lb, ub)
        evalObjCon(x) -> (fail, fobj, con)
        evalObjConGradient(x, g, A) -> fail          A: list of ncon tensors
        writeOutput(it, x)                           optional
        evalHvecProduct(x, z, zw, px, hvec) -> fail  optional; z: ncon host values
        evalHessianDiag(x, z, zw, hdiag) -> fail     optional (use_diag_hessian)
        computeQuasiNewtonUpdateCorrection(x, z, zw, s, y) -> fail   optional

    Every vector is a float64 CUDA tensor viewing the library's own memory: fill the
    outputs in place (g.copy_(...), A[j].copy_(...)); nothing is copied between host
    and device.  fobj and con may be Python floats, 0-d tensors or a 1-D tensor; they
    reach the host in one device->host copy per evalObjCon.  As in Problem, an
    optional callback is registered only when the subclass defines it.

    The callbacks run with torch's current stream set to the context's stream
    (Context.stream), after that stream has been made to wait on the stream that was
    current when the optimizer was called, so tensors filled just before optimize()
    are complete when a callback reads them.  Multi-rank problems reduce their
    partial sums with Context.allreduce_sum.

    `x` handed to different callbacks may be different buffers holding the same
    values (the optimizer exchanges vectors instead of copying them): do not cache
    results by tensor or pointer.

    An exception in a callback prints its traceback and reports a failed
    evaluation.  Later callbacks of the same run then fail without calling the
    subclass, and InteriorPoint / TrustRegion raise RuntimeError from the first
    exception when the run returns."""

    def __init__(self, ctx, nvars, ncon, ninequality=-1, nwinequality=-1,
                 use_lower=True, use_upper=True, weighting=None):
        import torch
        self.ctx = ctx
        self.lib = ctx.lib
        self.nvars, self.ncon = int(nvars), int(ncon)
        self.device = torch.device("cuda", ctx.device)
        w = _lib.Weighting()
        if weighting:
            for k, v in weighting.items():
                setattr(w, k, v)
        self._w = w
        self._views = {}
        self._error = None
        self._ready = None  # event: the caller's stream at the entry of a callback
        self._empty = torch.empty(0, dtype=torch.float64, device=self.device)
        cb = _lib.Callbacks()
        cb.user = None
        cb.get_vars_and_bounds = _lib.GET_VARS_CB(self._get_vars)
        cb.eval_obj_con = _lib.EVAL_OBJ_CB(self._eval_obj)
        cb.eval_obj_con_gradient = _lib.EVAL_GRAD_CB(self._eval_grad)
        if hasattr(self, "computeQuasiNewtonUpdateCorrection"):
            cb.qn_update_correction = _lib.QN_CORR_CB(self._qn_correction)
        if hasattr(self, "writeOutput"):
            cb.write_output = _lib.WRITE_OUT_CB(self._write_output)
        if hasattr(self, "evalHvecProduct"):
            cb.eval_hvec_product = _lib.HVEC_CB(self._eval_hvec)
        self._cb = cb
        self.h = self.lib.pcu_problem_create(
            ctx.h, self.nvars, self.ncon, int(ninequality), int(nwinequality),
            int(use_lower), int(use_upper), C.byref(self._w), C.byref(self._cb))
        if not self.h:
            raise RuntimeError("paropt_b200: problem creation failed")
        if hasattr(self, "evalHessianDiag"):
            self._hdiag_cb = _lib.HDIAG_CB(self._eval_hdiag)
            _check(self.lib.pcu_problem_set_hessian_diag(self.h, None, self._hdiag_cb),
                   "set_hessian_diag")

    def _vec(self, h):
        """Zero-copy tensor view of a pcu_vec, cached by handle and device pointer: the
        quasi-Newton memory exchanges buffers, so a handle can change its storage."""
        if not h:
            return self._empty
        ptr = int(self.lib.pcu_vec_device_ptr(h) or 0)
        key = (h, ptr)
        t = self._views.get(key)
        if t is None:
            import torch
            n = int(self.lib.pcu_vec_size(h))
            t = (torch.as_tensor(_DeviceArray(ptr, n), device=self.device)
                 if n > 0 and ptr else self._empty)
            self._views[key] = t
        return t

    def _call(self, fn, *args):
        """Runs one callback body on the context's stream; 0 / 1 for the library."""
        if self._error is not None:
            return 1
        import torch
        try:
            stream = self.ctx.stream
            cur = torch.cuda.current_stream(self.device)
            if cur != stream:
                if self._ready is None:
                    self._ready = torch.cuda.Event()
                self._ready.record(cur)
                stream.wait_event(self._ready)
            with torch.cuda.stream(stream):
                return int(fn(*args) or 0)
        except Exception as e:  # report, do not unwind through C (ParOpt.pyx:528-531)
            import traceback
            traceback.print_exc()
            self._error = e
            return 1

    def take_callback_error(self):
        """The exception a callback raised in the last run (None if none), cleared."""
        e, self._error = self._error, None
        return e

    def _get_vars(self, user, x, lb, ub):
        return self._call(lambda: self.getVarsAndBounds(self._vec(x), self._vec(lb),
                                                        self._vec(ub)))

    def _eval_obj(self, user, x, fobj, cons):
        def body():
            fail, f, con = self.evalObjCon(self._vec(x))
            vals = self._host_values(f, con)
            fobj[0] = vals[0]
            for i in range(self.ncon):
                cons[i] = vals[i + 1]
            return fail
        return self._call(body)

    def _host_values(self, f, con):
        """[fobj, con...] as host floats: tensor entries are gathered into one device
        buffer and copied to the host once."""
        import torch
        out = [None] * (self.ncon + 1)
        dev = []  # (slot, tensor)
        if torch.is_tensor(f):
            dev.append((0, f.reshape(1)))
        else:
            out[0] = float(f)
        if torch.is_tensor(con):
            if con.numel() != self.ncon:
                raise ValueError("evalObjCon returned %d constraints, expected %d"
                                 % (con.numel(), self.ncon))
            if self.ncon:
                dev.append((1, con.reshape(-1)))
        else:
            con = list(con) if con is not None else []
            if len(con) != self.ncon:
                raise ValueError("evalObjCon returned %d constraints, expected %d"
                                 % (len(con), self.ncon))
            for i, c in enumerate(con):
                if torch.is_tensor(c):
                    dev.append((i + 1, c.reshape(1)))
                else:
                    out[i + 1] = float(c)
        if dev:
            buf = torch.empty(self.ncon + 1, dtype=torch.float64, device=self.device)
            for slot, t in dev:
                buf[slot:slot + t.numel()].copy_(t)
            host = buf.cpu().tolist()  # the one synchronisation
            for slot, t in dev:
                out[slot:slot + t.numel()] = host[slot:slot + t.numel()]
        return out

    def _eval_grad(self, user, x, g, Ac):
        return self._call(lambda: self.evalObjConGradient(
            self._vec(x), self._vec(g), [self._vec(Ac[i]) for i in range(self.ncon)]))

    def _eval_hvec(self, user, x, z, zw, px, hvec):
        zz = np.array([z[i] for i in range(self.ncon)])
        return self._call(lambda: self.evalHvecProduct(
            self._vec(x), zz, self._vec(zw), self._vec(px), self._vec(hvec)))

    def _eval_hdiag(self, user, x, z, zw, hdiag):
        zz = np.array([z[i] for i in range(self.ncon)])
        return self._call(lambda: self.evalHessianDiag(
            self._vec(x), zz, self._vec(zw), self._vec(hdiag)))

    def _qn_correction(self, user, x, z, zw, s, y):
        zz = np.array([z[i] for i in range(self.ncon)])
        return self._call(lambda: self.computeQuasiNewtonUpdateCorrection(
            self._vec(x), zz, self._vec(zw), self._vec(s), self._vec(y)))

    def _write_output(self, user, it, x):
        return self._call(lambda: self.writeOutput(int(it), self._vec(x)))

    def callback_ms(self):
        """Device milliseconds spent inside the callbacks (events on the context's stream)."""
        return float(self.lib.pcu_problem_callback_ms(self.h))

    def transfer_bytes(self):
        a, b = C.c_int64(), C.c_int64()
        self.lib.pcu_problem_transfer_bytes(self.h, C.byref(a), C.byref(b))
        return a.value, b.value

    @property
    def h2d_bytes(self):
        return self.transfer_bytes()[0]

    @property
    def d2h_bytes(self):
        return self.transfer_bytes()[1]

    def free(self):
        if self.h:
            self._views.clear()
            self.lib.pcu_problem_destroy(self.h)
            self.h = None


class AutogradProblem(TorchProblem):
    """A TorchProblem whose derivatives come from torch.autograd: subclass and
    implement getVarsAndBounds(x, lb, ub) and objcon(x) -> (f, c) with f a 0-d tensor
    and c a 1-D tensor (or list) of the ncon constraints, written in differentiable
    torch operations.  The gradients are one backward pass per output through a
    retained graph; the Hessian-vector product (use_hvec_product) is the double
    backward of the Lagrangian L = f - z^T c (the reference's sign convention; the
    weighting rows are linear and add nothing)."""

    def _outputs(self, x):
        f, c = self.objcon(x)
        cs = [c[i] for i in range(self.ncon)]
        return f, cs

    def evalObjCon(self, x):
        import torch
        with torch.no_grad():
            f, c = self.objcon(x)
        return 0, f, c

    def evalObjConGradient(self, x, g, A):
        import torch
        with torch.enable_grad():
            xr = x.detach().requires_grad_(True)
            f, cs = self._outputs(xr)
            outs = [f] + cs
            for k, (out, dst) in enumerate(zip(outs, [g] + list(A))):
                grad = None
                if torch.is_tensor(out) and out.requires_grad:
                    (grad,) = torch.autograd.grad(out, xr, retain_graph=k + 1 < len(outs),
                                                  allow_unused=True)
                if grad is None:
                    dst.zero_()
                else:
                    dst.copy_(grad)
        return 0

    def evalHvecProduct(self, x, z, zw, px, hvec):
        import torch
        with torch.enable_grad():
            xr = x.detach().requires_grad_(True)
            f, cs = self._outputs(xr)
            L = f
            for zj, cj in zip(z, cs):
                L = L - float(zj) * cj
            hv = None
            if torch.is_tensor(L) and L.requires_grad:
                (gL,) = torch.autograd.grad(L, xr, create_graph=True)
                if gL.requires_grad:
                    (hv,) = torch.autograd.grad(gL, xr, grad_outputs=px, allow_unused=True)
            if hv is None:
                hvec.zero_()
            else:
                hvec.copy_(hv)
        return 0


def _raise_callback_error(prob, rc, what):
    """RuntimeError for a failed library call, chained to the exception a
    TorchProblem callback raised during it (the library may absorb a failed
    evaluation, e.g. by shortening a line-search step)."""
    take = getattr(prob, "take_callback_error", None)
    err = take() if take is not None else None
    if err is not None:
        raise RuntimeError("paropt_b200: %s: a problem callback raised %s: %s"
                           % (what, type(err).__name__, err)) from err
    _check(rc, what)


class BuiltinProblem:
    """Synthetic problems shipped with the library: GPU-resident
    (pcu_problem_create_sepquad / _rosenbrock) or, with host=True, the same
    sepquad workload as threaded C++ host callbacks over host arrays
    (pcu_problem_create_sepquad_host) -- the end-to-end path."""

    def __init__(self, ctx, kind, host=False, nthreads=0, **params):
        self.ctx = ctx
        self.lib = ctx.lib
        self._user = None
        if kind == "sepquad":
            self._p = sepquad_params(**params)
            if host:
                user = C.c_void_p()
                self.h = self.lib.pcu_problem_create_sepquad_host(
                    ctx.h, C.byref(self._p), int(nthreads), C.byref(user))
                self._user = user
            else:
                self.h = self.lib.pcu_problem_create_sepquad(ctx.h, C.byref(self._p))
        elif kind == "rosenbrock":
            n = int(params.get("n", 1000))
            self.h = self.lib.pcu_problem_create_rosenbrock(ctx.h, n - 1, 5, 1, 5, 1)
        else:
            raise ValueError(kind)
        if not self.h:
            raise RuntimeError("paropt_b200: problem creation failed")
        nv, nc, nw = C.c_int(), C.c_int(), C.c_int()
        self.lib.pcu_problem_sizes(self.h, C.byref(nv), C.byref(nc), C.byref(nw))
        self.nvars, self.ncon, self.nwcon = nv.value, nc.value, nw.value

    def callback_ms(self):
        return float(self.lib.pcu_problem_callback_ms(self.h))

    def transfer_bytes(self):
        a, b = C.c_int64(), C.c_int64()
        self.lib.pcu_problem_transfer_bytes(self.h, C.byref(a), C.byref(b))
        return a.value, b.value

    def host_times(self):
        """(d2h_ms, user_ms, h2d_ms) of a host-array problem (see the header)."""
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        self.lib.pcu_problem_host_times(self.h, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def free(self):
        if self.h:
            self.lib.pcu_problem_destroy(self.h)
            self.h = None
        if self._user is not None and self._user.value:
            self.lib.pcu_problem_sepquad_host_free(self._user)
            self._user = None


def problem_from_config(ctx, cfg):
    if cfg["kind"] == "rosenbrock":
        return BuiltinProblem(ctx, "rosenbrock", **cfg["problem"])
    return BuiltinProblem(ctx, "sepquad", **cfg["problem"])


class InteriorPoint:
    """ParOpt.InteriorPoint (ParOpt.pyx:1189-1365 / ParOptInteriorPoint.h:128)."""

    def __init__(self, problem, options=None):
        self.prob = problem
        self.ctx = problem.ctx
        self.lib = self.ctx.lib
        self.h = self.lib.pcu_ip_create(problem.h)
        if not self.h:
            raise RuntimeError("paropt_b200: interior-point creation failed")
        self.ncon = problem.ncon
        for k, v in (options or {}).items():
            self.setOption(k, v)

    def setOption(self, name, value):
        key = name.encode()
        if isinstance(value, bool):
            rc = self.lib.pcu_ip_set_option_int(self.h, key, int(value))
        elif isinstance(value, int):
            rc = self.lib.pcu_ip_set_option_int(self.h, key, value)
        elif isinstance(value, float):
            rc = self.lib.pcu_ip_set_option_float(self.h, key, value)
        else:
            rc = self.lib.pcu_ip_set_option_str(self.h, key, str(value).encode())
        if rc != 0:  # ParOpt.pyx:411-413 raises ValueError for unknown options
            raise ValueError("unknown or out-of-range option %s=%r" % (name, value))

    def setQuasiNewton(self, qn):
        """ParOptInteriorPoint::setQuasiNewton (IP.cpp:1193): use the caller's
        QuasiNewton object (None: the optimizer's own)."""
        _check(self.lib.pcu_ip_set_quasi_newton(self.h, qn.h if qn is not None else None),
               "setQuasiNewton")
        self._qn_ref = qn  # keep it alive

    def resetDesignAndBounds(self):
        """ParOptInteriorPoint::resetDesignAndBounds (IP.cpp:1249)."""
        _check(self.lib.pcu_ip_reset_design_and_bounds(self.h), "resetDesignAndBounds")

    def setPenaltyGamma(self, gamma):
        """setPenaltyGamma(double) / setPenaltyGamma(const double*) (IP.cpp:1128, 1160)."""
        if np.isscalar(gamma):
            _check(self.lib.pcu_ip_set_penalty_gamma(self.h, float(gamma)), "setPenaltyGamma")
        else:
            g = np.ascontiguousarray(gamma, dtype=np.float64)
            if g.size != self.ncon:
                raise ValueError("penalty array must have ncon entries")
            _check(self.lib.pcu_ip_set_penalty_gamma_array(
                self.h, g.ctypes.data_as(_lib.c_double_p)), "setPenaltyGamma")

    def getPenaltyGamma(self):
        g = np.zeros(max(self.ncon, 1))
        _check(self.lib.pcu_ip_get_penalty_gamma(self.h, g.ctypes.data_as(_lib.c_double_p)),
               "getPenaltyGamma")
        return g[:self.ncon]

    def resetProblemInstance(self, problem):
        """resetProblemInstance (IP.cpp:745): a congruent problem replaces the current one."""
        _check(self.lib.pcu_ip_reset_problem(self.h, problem.h), "resetProblemInstance")
        self.prob = problem

    def writeSolutionFile(self, filename):
        """ParOptInteriorPoint::writeSolutionFile (IP.cpp:883): the reference's binary layout."""
        return int(self.lib.pcu_ip_write_solution(self.h, str(filename).encode()))

    def readSolutionFile(self, filename):
        """ParOptInteriorPoint::readSolutionFile (IP.cpp:986)."""
        return int(self.lib.pcu_ip_read_solution(self.h, str(filename).encode()))

    def resetQuasiNewtonHessian(self):
        _check(self.lib.pcu_ip_reset_quasi_newton(self.h), "resetQuasiNewtonHessian")

    def optimize(self):
        _raise_callback_error(self.prob, self.lib.pcu_ip_optimize(self.h), "optimize")

    def begin(self):
        _raise_callback_error(self.prob, self.lib.pcu_ip_begin(self.h), "begin")

    def iterate(self, n=1):
        conv = C.c_int()
        _raise_callback_error(self.prob, self.lib.pcu_ip_iterate(self.h, int(n), C.byref(conv)),
                              "iterate")
        return bool(conv.value)

    def status(self):
        return STATUS[int(self.lib.pcu_ip_status(self.h))]

    def counters(self):
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        self.lib.pcu_ip_counters(self.h, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def getBarrierParameter(self):
        return float(self.lib.pcu_ip_barrier_param(self.h))

    def getComplementarity(self):
        out = C.c_double()
        _check(self.lib.pcu_ip_complementarity(self.h, C.byref(out)), "comp")
        return out.value

    def getOptimizedPoint(self):
        hs = [C.c_void_p() for _ in range(6)]
        self.lib.pcu_ip_get_point(self.h, *[C.byref(h) for h in hs])
        vecs = [PVec(self.ctx, handle=h.value) for h in hs]
        dense = self.get_dense()
        # reference order: x, z, zw, zl, zu
        return vecs[0], dense["z"], vecs[1], vecs[2], vecs[3]

    def get_dense(self):
        c = self.ncon
        arrs = {k: np.zeros(c) for k in ("z", "s", "t", "zs", "zt", "c")}
        self.lib.pcu_ip_get_dense(self.h, *[arrs[k].ctypes.data_as(_lib.c_double_p)
                                           for k in ("z", "s", "t", "zs", "zt", "c")])
        return arrs

    def history(self):
        n = int(self.lib.pcu_ip_history_len(self.h))
        c = self.ncon
        buf = np.zeros(len(HIST_FIELDS) + 6 * c)
        out = []
        for k in range(n):
            _check(self.lib.pcu_ip_history_get(self.h, k, buf.ctypes.data_as(_lib.c_double_p),
                                               buf.size), "history")
            rec = {name: float(buf[i]) for i, name in enumerate(HIST_FIELDS)}
            for name in ("iter", "neval", "ngeval", "qn_size", "nhvec"):
                rec[name] = int(rec[name])
            off = len(HIST_FIELDS)
            for j, name in enumerate(("c", "z", "s", "t", "zs", "zt")):
                rec[name] = buf[off + j * c: off + (j + 1) * c].tolist()
            rec["info"] = self.lib.pcu_ip_history_info(self.h, k).decode()
            out.append(rec)
        return out

    def iter_times(self):
        out = []
        k = 0
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        while self.lib.pcu_ip_iter_times(self.h, k, C.byref(a), C.byref(b), C.byref(c)) == 0:
            out.append((a.value, b.value, c.value))
            k += 1
        return out

    # ---- function-level access (kernel parity tests) -------------------
    def vars_vec(self, which, comp):
        h = self.lib.pcu_ip_vars_vec(self.h, which, comp)
        return PVec(self.ctx, handle=h)

    def state_vec(self, ident):
        return PVec(self.ctx, handle=self.lib.pcu_ip_state_vec(self.h, ident))

    def dense_get(self, which):
        buf = np.zeros(5 * self.ncon)
        self.lib.pcu_ip_vars_dense_get(self.h, which, buf.ctypes.data_as(_lib.c_double_p))
        c = self.ncon
        return {k: buf[i * c:(i + 1) * c].copy() for i, k in enumerate(("z", "s", "t", "zs", "zt"))}

    def dense_set(self, which, d):
        buf = np.concatenate([np.asarray(d[k], dtype=np.float64) for k in ("z", "s", "t", "zs", "zt")]) \
            if self.ncon else np.zeros(0)
        buf = np.ascontiguousarray(buf)
        self.lib.pcu_ip_vars_dense_set(self.h, which, buf.ctypes.data_as(_lib.c_double_p))

    def free(self):
        if self.h:
            self.lib.pcu_ip_destroy(self.h)
            self.h = None


TR_FIELDS = ("iter", "fobj", "infeas", "l1", "linfty", "dx", "tr", "rho", "model_red", "zav",
             "zmax", "gav", "gmax", "subproblem_iters", "adaptive_iters", "accepted", "xsum",
             "xnorm", "xmaxabs")


class TrustRegion:
    """ParOptTrustRegion + ParOptQuadraticSubproblem on the device (pcu_tr): the SL1QP
    penalty method with the adaptive penalty update (ParOptTrustRegion.cpp:1454-1690);
    what ParOpt.Optimizer runs for algorithm = "tr"."""

    def __init__(self, problem, options=None):
        self.prob = problem
        self.ctx = problem.ctx
        self.lib = self.ctx.lib
        self.h = self.lib.pcu_tr_create(problem.h)
        if not self.h:
            raise RuntimeError("paropt_b200: trust-region creation failed")
        self.ncon = problem.ncon
        for k, v in (options or {}).items():
            self.setOption(k, v)

    def setOption(self, name, value):
        key = name.encode()
        if isinstance(value, bool):
            rc = self.lib.pcu_tr_set_option_int(self.h, key, int(value))
        elif isinstance(value, int):
            rc = self.lib.pcu_tr_set_option_int(self.h, key, value)
        elif isinstance(value, float):
            rc = self.lib.pcu_tr_set_option_float(self.h, key, value)
        else:
            rc = self.lib.pcu_tr_set_option_str(self.h, key, str(value).encode())
        if rc != 0:
            raise ValueError("option %s=%r is not available" % (name, value))

    def optimize(self):
        _raise_callback_error(self.prob, self.lib.pcu_tr_optimize(self.h),
                              "trust-region optimize")

    def converged(self):
        return int(self.lib.pcu_tr_status(self.h)) == 1

    def history(self):
        out = []
        buf = np.zeros(len(TR_FIELDS))
        for k in range(int(self.lib.pcu_tr_history_len(self.h))):
            _check(self.lib.pcu_tr_history_get(self.h, k, buf.ctypes.data_as(_lib.c_double_p)),
                   "tr history")
            rec = {name: float(buf[i]) for i, name in enumerate(TR_FIELDS)}
            for name in ("iter", "subproblem_iters", "adaptive_iters", "accepted"):
                rec[name] = int(rec[name])
            rec["info"] = self.lib.pcu_tr_history_info(self.h, k).decode()
            out.append(rec)
        return out

    def getOptimizedPoint(self):
        """x (the centre), z, zw, zl, zu of the last subproblem solve
        (ParOptOptimizer::getOptimizedPoint, ParOptOptimizer.cpp:231-262)."""
        x = PVec(self.ctx, handle=self.lib.pcu_tr_point(self.h))
        ip = InteriorPoint.__new__(InteriorPoint)
        ip.prob, ip.ctx, ip.lib, ip.ncon = self.prob, self.ctx, self.lib, self.ncon
        ip.h = self.lib.pcu_tr_interior_point(self.h)
        _, z, zw, zl, zu = ip.getOptimizedPoint()
        return x, z, zw, zl, zu

    def getPenaltyGamma(self):
        g = np.zeros(max(self.ncon, 1))
        self.lib.pcu_tr_penalty_gamma(self.h, g.ctypes.data_as(_lib.c_double_p))
        return g[:self.ncon]

    def free(self):
        if self.h:
            self.lib.pcu_tr_destroy(self.h)
            self.h = None
