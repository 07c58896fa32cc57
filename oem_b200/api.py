"""Host-side mirror of the reference's five C++ entry points, bound to liboem_b200.so through ctypes.

Same names, argument order and return layout as the reference's .Call interface
(R/oem.R:556-575, R/oem_xtx.R:389-420, R/oem_xval.R:525-548, R/big_oem.R:449-490, and the
RcppExport functions src/oem_dense.cpp:30, oem_xtx.cpp:29, oem_xval_dense.cpp:31,
oem_logistic_dense.cpp:29, oem_big.cpp:30):

    oem_fit_dense(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_,
                  nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                  compute_loss, opts)  ->  dict(beta=[...], lambda_=[...], niter=[...], loss=[...], d=...)

`x` / `y` may be numpy arrays (host; copied to the GPU inside the call) or torch CUDA tensors
(device; used in place - x must be column-major, i.e. x.stride() == (1, ld)).  There is no CPU
implementation behind these functions: without the CUDA library / a GPU they raise.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "lib", "liboem_b200.so")
_lib = None

ALLREDUCE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p)


class OemB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[oem_b200 error {code}] {msg}")
        self.code = code


class Opts(ctypes.Structure):
    _fields_ = [("maxit", ctypes.c_int), ("tol", ctypes.c_double), ("irls_maxit", ctypes.c_int),
                ("irls_tol", ctypes.c_double), ("ncores", ctypes.c_int), ("hessian_full", ctypes.c_int),
                ("accelerate", ctypes.c_int), ("gigs", ctypes.c_double), ("device", ctypes.c_int),
                ("stream", ctypes.c_void_p), ("allreduce", ALLREDUCE_FN), ("allreduce_ctx", ctypes.c_void_p),
                ("rank", ctypes.c_int), ("world", ctypes.c_int), ("comm", ctypes.c_void_p)]


class Spec(ctypes.Structure):
    _fields_ = [("family", ctypes.c_char_p), ("n_penalty", ctypes.c_int),
                ("penalty", ctypes.POINTER(ctypes.c_char_p)),
                ("weights", ctypes.c_void_p), ("n_weights", ctypes.c_int64),
                ("groups", ctypes.c_void_p), ("n_groups", ctypes.c_int),
                ("unique_groups", ctypes.c_void_p), ("n_unique_groups", ctypes.c_int),
                ("group_weights", ctypes.c_void_p), ("n_group_weights", ctypes.c_int),
                ("lambda_", ctypes.POINTER(ctypes.c_void_p)), ("n_lambda", ctypes.c_void_p),
                ("nlambda", ctypes.c_int), ("lambda_min_ratio", ctypes.c_double), ("alpha", ctypes.c_double),
                ("gamma", ctypes.c_void_p), ("n_gamma", ctypes.c_int), ("tau", ctypes.c_double),
                ("penalty_factor", ctypes.c_void_p), ("standardize", ctypes.c_int), ("intercept", ctypes.c_int),
                ("compute_loss", ctypes.c_int)]


class Stats(ctypes.Structure):
    _fields_ = [(k, ctypes.c_double) for k in
                ("ms_h2d", "ms_colstats", "ms_gram", "ms_gram_reduce", "ms_allreduce", "ms_assemble", "ms_path",
                 "ms_cvscore", "ms_irls_xb", "ms_irls_xtr", "ms_total", "gram_flops", "gemv_bytes")] + \
               [(k, ctypes.c_int64) for k in
                ("kernel_launches", "gram_launches", "xb_launches", "xtr_launches", "total_oem_iters",
                 "lanczos_steps", "h2d_bytes", "d2h_bytes", "allreduce_calls", "allreduce_doubles", "data_passes",
                 "host_syncs")] + \
               [(k, ctypes.c_double) for k in ("ms_relayout", "ms_ingest_wait")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Result(ctypes.Structure):
    _fields_ = [("beta", ctypes.c_void_p), ("lambda_", ctypes.c_void_p), ("niter", ctypes.c_void_p),
                ("loss", ctypes.c_void_p), ("d", ctypes.c_void_p), ("cvm", ctypes.c_void_p),
                ("cvsd", ctypes.c_void_p), ("nlam_out", ctypes.c_void_p), ("stats", ctypes.POINTER(Stats))]


def lib_path():
    return _LIB_PATH


def load():
    """Load liboem_b200.so; fails loudly when the CUDA library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("OEMB200_LIB_PATH", _LIB_PATH)      # A/B runs of two builds of the same ABI (tools/ab_build.sh)
    if not os.path.exists(path):
        raise OemB200Error(-1, f"{path} is missing: run `python -m oem_b200.build` "
                               "(the CUDA extension is the only implementation; there is no CPU fallback)")
    L = ctypes.CDLL(path)
    L.oemb200_last_error.restype = ctypes.c_char_p
    L.oemb200_version.restype = ctypes.c_char_p
    L.oemb200_device_count.restype = ctypes.c_int
    L.oemb200_default_opts.argtypes = [ctypes.POINTER(Opts)]
    L.oemb200_penalty_id.argtypes = [ctypes.c_char_p]
    L.oemb200_nlambda_max.argtypes = [ctypes.POINTER(Spec)]
    vp, i64, ci, dbl = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double
    sp, op, rp = ctypes.POINTER(Spec), ctypes.POINTER(Opts), ctypes.POINTER(Result)
    L.oemb200_fit_dense.argtypes = [vp, i64, ci, i64, vp, sp, op, rp]
    L.oemb200_fit_big.argtypes = [vp, i64, ci, i64, vp, sp, op, rp]
    L.oemb200_fit_sparse.argtypes = [vp, vp, vp, i64, ci, vp, sp, op, rp]
    L.oemb200_fit_logistic_sparse.argtypes = [vp, vp, vp, i64, ci, vp, sp, op, rp]
    L.oemb200_fit_logistic_dense.argtypes = [vp, i64, ci, i64, vp, sp, op, rp]
    L.oemb200_xtx.argtypes = [vp, vp, ci, sp, vp, ci, op, rp]
    L.oemb200_xval_dense.argtypes = [vp, i64, ci, i64, vp, sp, ci, vp, ctypes.c_char_p, op, rp]
    L.oemb200_xval_logistic_dense.argtypes = [vp, i64, ci, i64, vp, sp, ci, vp, ctypes.c_char_p, op, rp]
    L.oemb200_xval_big.argtypes = [vp, i64, ci, i64, vp, sp, ci, vp, ctypes.c_char_p, op, rp]
    L.oemb200_xval_logistic_dense_h.argtypes = [vp, vp, sp, ci, vp, ctypes.c_char_p, op, rp]
    L.oemb200_logit_fold_pass.argtypes = [vp, i64, ci, i64, vp, vp, vp, vp, ci, vp, vp, ci, vp, ctypes.POINTER(dbl),
                                          ctypes.POINTER(dbl), ctypes.POINTER(ci)]
    L.oemb200_gram.argtypes = [vp, i64, ci, i64, vp, vp, vp, vp, ctypes.POINTER(dbl)]
    L.oemb200_colstats.argtypes = [vp, i64, ci, i64, vp, vp, vp, vp, ctypes.POINTER(dbl)]
    L.oemb200_xb_logistic.argtypes = [vp, i64, ci, i64, vp, dbl, vp, vp, vp, vp, vp, ctypes.POINTER(dbl)]
    L.oemb200_top_eig.argtypes = [vp, ci, ctypes.POINTER(dbl), ctypes.POINTER(ci), vp]
    L.oemb200_logit_slab_pass.argtypes = [vp, i64, ci, i64, vp, dbl, vp, vp, vp, vp, ci, vp, ctypes.POINTER(dbl),
                                          ctypes.POINTER(dbl)]
    L.oemb200_matrix_create.argtypes = [vp, i64, ci, i64, op, ctypes.POINTER(vp)]
    L.oemb200_matrix_create_from_file.argtypes = [ctypes.c_char_p, i64, ci, op, ctypes.POINTER(vp)]
    L.oemb200_matrix_destroy.argtypes = [vp]
    L.oemb200_matrix_info.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(ci), ctypes.POINTER(i64), ctypes.POINTER(vp),
                                      ctypes.POINTER(i64), ctypes.POINTER(dbl)]
    L.oemb200_fit_dense_h.argtypes = [vp, vp, sp, op, rp]
    L.oemb200_fit_big_h.argtypes = [vp, vp, sp, op, rp]
    L.oemb200_fit_logistic_dense_h.argtypes = [vp, vp, sp, op, rp]
    L.oemb200_xval_dense_h.argtypes = [vp, vp, sp, ci, vp, ctypes.c_char_p, op, rp]
    L.oemb200_predict_h.argtypes = [vp, vp, ci, ci, ci, vp, i64, op, ctypes.POINTER(Stats)]
    L.oemb200_comm_unique_id.argtypes = [vp]
    L.oemb200_comm_create.argtypes = [vp, ci, ci, ci, ctypes.POINTER(vp)]
    L.oemb200_comm_from_nccl.argtypes = [vp, ci, ci, ci, ctypes.POINTER(vp)]
    L.oemb200_comm_destroy.argtypes = [vp]
    L.oemb200_comm_allreduce.argtypes = [vp, vp, i64, vp, ctypes.POINTER(dbl)]
    L.oemb200_comm_p2p_enabled.argtypes = [vp]
    L.oemb200_lambda_grid.argtypes = [dbl, ci, dbl, vp]
    L.oemb200_stop_rule.argtypes = [vp, vp, ci, dbl]
    L.oemb200_release_cache.restype = None
    L.oemb200_predict.argtypes = [vp, i64, ci, i64, vp, ci, ci, ci, vp, i64, op, ctypes.POINTER(Stats)]
    L.oemb200_predict_sparse.argtypes = [vp, vp, vp, i64, ci, vp, ci, ci, ci, vp, i64, op, ctypes.POINTER(Stats)]
    _lib = L
    return L


EXPORTS = ["oemb200_last_error", "oemb200_version", "oemb200_device_count", "oemb200_default_opts",
           "oemb200_penalty_id", "oemb200_nlambda_max", "oemb200_fit_dense", "oemb200_xtx", "oemb200_xval_dense",
           "oemb200_fit_logistic_dense", "oemb200_fit_big", "oemb200_fit_sparse", "oemb200_fit_logistic_sparse", "oemb200_gram", "oemb200_colstats",
           "oemb200_xb_logistic", "oemb200_top_eig", "oemb200_lambda_grid", "oemb200_stop_rule",
           "oemb200_release_cache", "oemb200_predict", "oemb200_predict_sparse", "oemb200_logit_slab_pass",
           "oemb200_matrix_create", "oemb200_matrix_create_from_file", "oemb200_matrix_destroy", "oemb200_matrix_info",
           "oemb200_fit_dense_h", "oemb200_fit_big_h", "oemb200_fit_logistic_dense_h", "oemb200_xval_dense_h",
           "oemb200_predict_h", "oemb200_comm_unique_id", "oemb200_comm_create", "oemb200_comm_from_nccl", "oemb200_comm_destroy",
           "oemb200_comm_allreduce", "oemb200_comm_p2p_enabled", "oemb200_xval_logistic_dense",
           "oemb200_xval_logistic_dense_h", "oemb200_logit_fold_pass", "oemb200_xval_big"]


def lambda_grid(lmax, nlambda, lmin_ratio):
    """Host-side lambda grid of the library (src/oem_dense.cpp:179-186)."""
    out = np.zeros(int(nlambda))
    _check(load().oemb200_lambda_grid(float(lmax), int(nlambda), float(lmin_ratio), out.ctypes.data))
    return out


def stop_rule(cur, prev, tol):
    cur = np.ascontiguousarray(cur, dtype=np.float64)
    prev = np.ascontiguousarray(prev, dtype=np.float64)
    return bool(load().oemb200_stop_rule(cur.ctypes.data, prev.ctypes.data, cur.size, float(tol)))


def _check(rc):
    if rc != 0:
        raise OemB200Error(rc, load().oemb200_last_error().decode())


def _is_torch_cuda(a):
    return type(a).__module__.startswith("torch") and getattr(a, "is_cuda", False)


class DeviceMatrix:
    """Device-resident design matrix (oemb200_matrix_*): uploaded once, then passed as `x` to oem_fit_dense / oem_fit_big /
    oem_fit_logistic_dense / oem_xval_dense / predict_matrix, which run on it without re-uploading.  `x` is a numpy array /
    np.memmap (host), a column-major CUDA tensor (copied on the device), or the path of a bigmemory backing file (.bk: raw
    column-major doubles) together with shape=(n, p)."""

    def __init__(self, x, shape=None, opts=None):
        L = load()
        o = opts if isinstance(opts, Opts) else make_opts(opts)
        h = ctypes.c_void_p()
        if isinstance(x, (str, bytes, os.PathLike)):
            if shape is None:
                raise ValueError("shape=(n, p) is required with a backing-file path")
            _check(L.oemb200_matrix_create_from_file(os.fsencode(x), int(shape[0]), int(shape[1]), ctypes.byref(o), ctypes.byref(h)))
        else:
            keep = _Keep()
            xp, n, p, ld = _matrix_arg(x, keep)
            _check(L.oemb200_matrix_create(xp, n, p, ld, ctypes.byref(o), ctypes.byref(h)))
        self.handle = h.value
        n, p, ld, ptr, nb, ms = ctypes.c_int64(), ctypes.c_int(), ctypes.c_int64(), ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_double()
        _check(L.oemb200_matrix_info(self.handle, ctypes.byref(n), ctypes.byref(p), ctypes.byref(ld), ctypes.byref(ptr),
                                     ctypes.byref(nb), ctypes.byref(ms)))
        self.shape = (n.value, p.value)
        self.ld, self.data_ptr, self.h2d_bytes, self.ms_upload = ld.value, ptr.value, nb.value, ms.value

    def close(self):
        if getattr(self, "handle", None):
            load().oemb200_matrix_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Keep:
    """Keeps the numpy temporaries backing raw pointers alive for the duration of a call."""

    def __init__(self):
        self.refs = []

    def arr(self, a, dtype):
        a = np.ascontiguousarray(np.asarray(a, dtype=dtype).ravel())
        self.refs.append(a)
        return a

    def ptr(self, a, dtype):
        a = self.arr(a, dtype)
        return a.ctypes.data if a.size else None, a.size


def _matrix_arg(x, keep):
    """-> (pointer, n, p, ld) for a column-major matrix on host (numpy), on device (torch) or held by a DeviceMatrix."""
    if isinstance(x, DeviceMatrix):
        if not x.handle:
            raise ValueError("DeviceMatrix has been closed")
        keep.refs.append(x)
        return x.data_ptr, x.shape[0], x.shape[1], x.ld
    if _is_torch_cuda(x):
        import torch
        if x.dtype != torch.float64 or x.dim() != 2:
            raise ValueError("device x must be a 2-D float64 tensor")
        n, p = x.shape
        if x.stride(0) != 1 and n > 1:
            raise ValueError("device x must be column-major (stride (1, ld)); e.g. torch.empty(p, n).t()")
        ld = x.stride(1) if p > 1 else n
        keep.refs.append(x)
        return x.data_ptr(), n, p, max(ld, n)
    a = np.asfortranarray(np.asarray(x, dtype=np.float64))
    if a.ndim != 2:
        raise ValueError("x must be 2-D")
    keep.refs.append(a)
    return a.ctypes.data, a.shape[0], a.shape[1], a.shape[0]


def _vector_arg(y, keep):
    if _is_torch_cuda(y):
        import torch
        if y.dtype != torch.float64:
            raise ValueError("device y must be float64")
        y = y.contiguous().view(-1)
        keep.refs.append(y)
        return y.data_ptr(), y.numel()
    a = keep.arr(y, np.float64)
    return a.ctypes.data, a.size


def make_opts(opts=None, comm=None):
    """Reference `options` list (R/oem.R:438-444) -> Opts.  Keys use '_' or '.'; extra runtime
    keys: device, stream.  `comm` is a oem_b200.dist.Comm (row-sharded multi-process runs)."""
    o = Opts()
    load().oemb200_default_opts(ctypes.byref(o))
    for k, v in (opts or {}).items():
        k = k.replace(".", "_")
        if k == "hessian_type":
            o.hessian_full = 1 if v == "full" else 0
        elif k in ("maxit", "irls_maxit", "ncores", "device"):
            setattr(o, k, int(v))
        elif k in ("tol", "irls_tol", "gigs"):
            setattr(o, k, float(v))
        elif k == "accelerate":
            o.accelerate = int(bool(v))
        elif k == "stream":
            o.stream = int(v)
        else:
            raise ValueError(f"unknown option {k}")
    if comm is not None and comm.world > 1:
        if getattr(comm, "handle", None):           # oem_b200.dist.LibComm: the library all-reduces by itself
            o.comm = comm.handle
        else:                                       # oem_b200.dist.Comm: host callback (torch.distributed)
            o.allreduce = comm.callback
        o.rank, o.world = comm.rank, comm.world
    return o


def _make_spec(keep, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
               lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss):
    s = Spec()
    s.family = family.encode()
    pens = [p.encode() for p in penalty]
    arr = (ctypes.c_char_p * len(pens))(*pens)
    keep.refs.append(arr)
    s.n_penalty = len(pens)
    s.penalty = arr
    s.weights, s.n_weights = keep.ptr(weights if weights is not None else [], np.float64)
    s.groups, s.n_groups = keep.ptr(groups if groups is not None else [], np.int32)
    s.unique_groups, s.n_unique_groups = keep.ptr(unique_groups if unique_groups is not None else [], np.int32)
    s.group_weights, s.n_group_weights = keep.ptr(group_weights if group_weights is not None else [], np.float64)
    lam_list = list(lambda_) if lambda_ is not None else []
    given = len(lam_list) > 0 and np.asarray(lam_list[0]).size >= 1
    if given:
        if len(lam_list) != len(pens):
            raise ValueError("lambda must be a list with one vector per penalty")
        ptrs = (ctypes.c_void_p * len(pens))()
        lens = np.zeros(len(pens), dtype=np.int32)
        for i, lv in enumerate(lam_list):
            a = keep.arr(lv, np.float64)
            ptrs[i] = a.ctypes.data
            lens[i] = a.size
        keep.refs += [ptrs, lens]
        s.lambda_ = ptrs
        s.n_lambda = lens.ctypes.data
    s.nlambda = int(nlambda)
    s.lambda_min_ratio = float(lmin_ratio)
    s.alpha = float(alpha)
    s.gamma, s.n_gamma = keep.ptr(np.atleast_1d(gamma), np.float64)
    s.tau = float(tau)
    s.penalty_factor, _ = keep.ptr(penalty_factor, np.float64)
    s.standardize = int(bool(standardize))
    s.intercept = int(bool(intercept))
    s.compute_loss = int(bool(compute_loss))
    return s


class _Out:
    def __init__(self, P, L, rows, xval=False):
        self.P, self.L, self.rows = P, L, rows
        self.beta = np.zeros((P, L, rows))
        self.lam = np.zeros((P, L))
        self.niter = np.zeros((P, L), dtype=np.int32)
        self.loss = np.zeros((P, L))
        self.d = np.zeros(1)
        self.cvm = np.zeros((P, L)) if xval else None
        self.cvsd = np.zeros((P, L)) if xval else None
        self.nlam = np.zeros(P, dtype=np.int32)
        self.stats = Stats()
        r = Result()
        r.beta, r.lambda_, r.niter = self.beta.ctypes.data, self.lam.ctypes.data, self.niter.ctypes.data
        r.loss, r.d, r.nlam_out = self.loss.ctypes.data, self.d.ctypes.data, self.nlam.ctypes.data
        if xval:
            r.cvm, r.cvsd = self.cvm.ctypes.data, self.cvsd.ctypes.data
        r.stats = ctypes.pointer(self.stats)
        self.res = r

    def as_dict(self):
        out = dict(beta=[], lambda_=[], niter=[], loss=[], d=float(self.d[0]), stats=self.stats.as_dict())
        for pp in range(self.P):
            k = int(self.nlam[pp])
            out["beta"].append(np.asfortranarray(self.beta[pp, :k, :].T))      # rows x k, column-major
            out["lambda_"].append(self.lam[pp].copy())
            out["niter"].append(self.niter[pp, :k].copy())
            out["loss"].append(self.loss[pp, :k].copy())
        if self.cvm is not None:
            out["cvm"] = [self.cvm[pp, :int(self.nlam[pp])].copy() for pp in range(self.P)]
            out["cvsd"] = [self.cvsd[pp, :int(self.nlam[pp])].copy() for pp in range(self.P)]
        return out


def _run_xy(fn_name, x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
            lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss, opts, comm,
            extra=None):
    L = load()
    keep = _Keep()
    handle = isinstance(x, DeviceMatrix) and fn_name != "oemb200_xval_big"
    if handle:
        if not x.handle:
            raise ValueError("DeviceMatrix has been closed")
        (n, p), xargs = x.shape, [x.handle]
        fn_name += "_h"
    else:
        xp, n, p, ld = _matrix_arg(x, keep)
        xargs = [xp, n, p, ld]
    yp, ny = _vector_arg(y, keep)
    if ny != n:
        raise ValueError("length of y must equal nrow(x)")
    spec = _make_spec(keep, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                      lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss)
    o = opts if isinstance(opts, Opts) else make_opts(opts, comm)
    Lmax = L.oemb200_nlambda_max(ctypes.byref(spec))
    out = _Out(len(penalty), Lmax, p + 1,
               xval=fn_name.startswith(("oemb200_xval_dense", "oemb200_xval_logistic_dense", "oemb200_xval_big")))
    fn = getattr(L, fn_name)
    if extra is None:
        rc = fn(*xargs, yp, ctypes.byref(spec), ctypes.byref(o), ctypes.byref(out.res))
    else:
        rc = fn(*xargs, yp, ctypes.byref(spec), *extra(keep), ctypes.byref(o), ctypes.byref(out.res))
    _check(rc)
    return out.as_dict()


def oem_fit_dense(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                  lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss, opts,
                  comm=None):
    """src/oem_dense.cpp:30-309."""
    return _run_xy("oemb200_fit_dense", x, y, family, penalty, weights, groups, unique_groups, group_weights,
                   lambda_, nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                   compute_loss, opts, comm)


def oem_fit_big(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss, opts,
                comm=None):
    """src/oem_big.cpp:30-258 (x = the big.matrix payload: n x p column-major doubles)."""
    return _run_xy("oemb200_fit_big", x, y, family, penalty, weights, groups, unique_groups, group_weights,
                   lambda_, nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                   compute_loss, opts, comm)


def _csc_slots(x):
    """(i, p, x, n, ncol) of a dgCMatrix-like input: a scipy.sparse matrix (converted to CSC with sorted, summed
    entries like as(x, "CsparseMatrix"), R/oem.R:240) or a tuple (i, p, x, (n, ncol)) of numpy arrays / CUDA tensors."""
    if isinstance(x, tuple):
        ri, cp, vals, (n, ncol) = x
        return ri, cp, vals, int(n), int(ncol)
    import scipy.sparse as sps
    if not sps.issparse(x):
        raise ValueError("oem_fit_sparse needs a scipy.sparse matrix or the (i, p, x, dim) slots of a dgCMatrix")
    c = sps.csc_matrix(x, dtype=np.float64)
    c.sum_duplicates()
    if c.nnz >= 2 ** 31:
        raise ValueError("more than 2^31 - 1 stored entries (the dgCMatrix limit)")
    return c.indices.astype(np.int32, copy=False), c.indptr.astype(np.int32, copy=False), c.data, c.shape[0], c.shape[1]


def _int_array_arg(a, keep):
    if _is_torch_cuda(a):
        import torch
        if a.dtype != torch.int32:
            raise ValueError("device index arrays must be int32")
        a = a.contiguous().view(-1)
        keep.refs.append(a)
        return a.data_ptr()
    a = keep.arr(a, np.int32)
    return a.ctypes.data if a.size else None


def oem_fit_logistic_sparse(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                            lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss, opts,
                            comm=None):
    """src/oem_logistic_sparse.cpp:30-330 (x = dgCMatrix: scipy.sparse matrix or its (i, p, x, dim) slots)."""
    return oem_fit_sparse(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                          lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss, opts,
                          comm=comm, _entry="oemb200_fit_logistic_sparse")


def oem_fit_sparse(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                   lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss, opts,
                   comm=None, _entry="oemb200_fit_sparse"):
    """src/oem_sparse.cpp:30-264 (x = dgCMatrix: scipy.sparse matrix or its (i, p, x, dim) slots)."""
    L = load()
    keep = _Keep()
    ri, cp, vals, n, p = _csc_slots(x)
    rip, cpp = _int_array_arg(ri, keep), _int_array_arg(cp, keep)
    vp_, _ = _vector_arg(vals, keep) if (_is_torch_cuda(vals) or np.asarray(vals).size) else (None, 0)
    yp, ny = _vector_arg(y, keep)
    if ny != n:
        raise ValueError("length of y must equal nrow(x)")
    spec = _make_spec(keep, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                      lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, compute_loss)
    o = opts if isinstance(opts, Opts) else make_opts(opts, comm)
    Lmax = L.oemb200_nlambda_max(ctypes.byref(spec))
    out = _Out(len(penalty), Lmax, p + 1, xval=False)
    _check(getattr(L, _entry)(rip, cpp, vp_, n, p, yp, ctypes.byref(spec), ctypes.byref(o), ctypes.byref(out.res)))
    return out.as_dict()


def oem_fit_logistic_dense(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_,
                           nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                           compute_loss, opts, comm=None):
    """src/oem_logistic_dense.cpp:29-313."""
    return _run_xy("oemb200_fit_logistic_dense", x, y, family, penalty, weights, groups, unique_groups,
                   group_weights, lambda_, nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize,
                   intercept, compute_loss, opts, comm)


def oem_xval_dense(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                   lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, nfolds, foldid,
                   compute_loss, type_measure, opts, comm=None):
    """src/oem_xval_dense.cpp:31-477."""
    def extra(keep):
        f = keep.arr(foldid, np.int32)
        return [int(nfolds), f.ctypes.data, type_measure.encode()]
    return _run_xy("oemb200_xval_dense", x, y, family, penalty, weights, groups, unique_groups, group_weights,
                   lambda_, nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                   compute_loss, opts, comm, extra=extra)


def oem_xval_big(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                 lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, nfolds, foldid,
                 compute_loss, type_measure, opts, comm=None):
    """oem_xval_dense on an x that is never resident on the device (include/oem_b200.h: oemb200_xval_big): x is read
    in row chunks of opts["gigs"] GB, once to form the fold Grams and once to score the fold models.  x is a numpy
    array, an np.memmap (e.g. oem_b200.bigmatrix.attach of a .bk file; pinned memory is copied without staging), a
    column-major CUDA tensor or a DeviceMatrix (read in place, no fold-sorted copy).  Gaussian family, one GPU."""
    def extra(keep):
        return [int(nfolds), _int_array_arg(foldid, keep), type_measure.encode()]
    return _run_xy("oemb200_xval_big", x, y, family, penalty, weights, groups, unique_groups, group_weights,
                   lambda_, nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                   compute_loss, opts, comm, extra=extra)


def oem_xval_logistic_dense(x, y, family, penalty, weights, groups, unique_groups, group_weights, lambda_, nlambda,
                            lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept, nfolds, foldid,
                            compute_loss, type_measure, opts, comm=None):
    """Binomial cross-validation (include/oem_b200.h: oemb200_xval_logistic_dense): the full-data logistic fit plus
    nfolds leave-fold-out fits at its lambdas, all IRLS passes fused; type_measure deviance | class | mse | mae."""
    def extra(keep):
        f = keep.arr(foldid, np.int32)
        return [int(nfolds), f.ctypes.data, type_measure.encode()]
    return _run_xy("oemb200_xval_logistic_dense", x, y, family, penalty, weights, groups, unique_groups, group_weights,
                   lambda_, nlambda, lmin_ratio, alpha, gamma, tau, penalty_factor, standardize, intercept,
                   compute_loss, opts, comm, extra=extra)


def logit_fold_pass(x, B, b0, y, fold, conv=None, reps=1, stream=None):
    """Phase-level fused data pass of the binomial xval (oemb200_logit_fold_pass) on CUDA tensors: x (n x p,
    column-major float64), B (M x p), b0 (M), y (n), fold (n, int32; 0 = no model), conv (M, int32, optional).
    Returns (grad M x (p + 1), ms per pass, ms of the slab re-layout, sweeps per pass)."""
    import torch
    keep = _Keep()
    xp, n, p, ld = _matrix_arg(x, keep)
    M = int(B.shape[0])
    for name, t, dt in (("B", B, torch.float64), ("b0", b0, torch.float64), ("y", y, torch.float64), ("fold", fold, torch.int32)):
        if not _is_torch_cuda(t) or t.dtype != dt or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous CUDA tensor of {dt}")
    if conv is not None and (not _is_torch_cuda(conv) or conv.dtype != torch.int32):
        raise ValueError("conv must be a CUDA int32 tensor")
    grad = torch.full((M, p + 1), float("nan"), dtype=torch.float64, device=B.device)
    ms, msr, sw = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
    _check(load().oemb200_logit_fold_pass(xp, n, p, ld, B.data_ptr(), b0.data_ptr(), y.data_ptr(), fold.data_ptr(), M,
                                          conv.data_ptr() if conv is not None else None, grad.data_ptr(), int(reps),
                                          stream, ctypes.byref(ms), ctypes.byref(msr), ctypes.byref(sw)))
    return grad, ms.value, msr.value, sw.value


def oem_xtx(xtx, xty, family, penalty, groups, unique_groups, group_weights, lambda_, nlambda, lmin_ratio,
            alpha, gamma, tau, scale_factor, penalty_factor, opts):
    """src/oem_xtx.cpp:29-219.  beta is p x nlambda (no intercept row)."""
    L = load()
    keep = _Keep()
    xp, p, p2, ld = _matrix_arg(xtx, keep)
    if p != p2 or ld != p:
        raise ValueError("xtx must be a dense square matrix")
    yp, ny = _vector_arg(xty, keep)
    if ny != p:
        raise ValueError("xty must have length ncol(xtx)")
    spec = _make_spec(keep, family, penalty, [], groups, unique_groups, group_weights, lambda_, nlambda,
                      lmin_ratio, alpha, gamma, tau, penalty_factor, False, False, False)
    o = opts if isinstance(opts, Opts) else make_opts(opts)
    Lmax = L.oemb200_nlambda_max(ctypes.byref(spec))
    out = _Out(len(penalty), Lmax, p)
    sfp, nsf = keep.ptr(scale_factor if scale_factor is not None else [], np.float64)
    _check(L.oemb200_xtx(xp, yp, p, ctypes.byref(spec), sfp, nsf, ctypes.byref(o), ctypes.byref(out.res)))
    return out.as_dict()


def predict_matrix(newx, beta, response=False, opts=None, out=None, return_stats=False):
    """newx %*% beta (+ intercept row) on the device: the GEMM of predict.oem (R/methods.R:113-118); response=True
    applies the logistic link of predict.oemfit_binomial (R/methods.R:355-358).  newx: n x p host (numpy) or device
    (column-major torch) matrix, or sparse (scipy.sparse / dgCMatrix slots -> oemb200_predict_sparse); beta: (p+1) x L with the intercept in row 0, or p x L.  Returns an n x L
    column-major numpy array, or fills `out` (a column-major float64 cuda tensor n x L) in place."""
    L = load()
    keep = _Keep()
    sparse = isinstance(newx, tuple) or type(newx).__module__.startswith("scipy.sparse")
    handle = isinstance(newx, DeviceMatrix)
    if handle:
        n, p = newx.shape
    elif sparse:
        ri, cp, vals, n, p = _csc_slots(newx)
        rip, cpp = _int_array_arg(ri, keep), _int_array_arg(cp, keep)
        vp_, _ = _vector_arg(vals, keep) if (_is_torch_cuda(vals) or np.asarray(vals).size) else (None, 0)
    else:
        xp, n, p, ld = _matrix_arg(newx, keep)
    b = np.asfortranarray(np.asarray(beta, dtype=np.float64))
    if b.ndim == 1:
        b = b.reshape(-1, 1, order="F")
    rows, nl = b.shape
    o = opts if isinstance(opts, Opts) else make_opts(opts, None)
    st = Stats()
    if out is None:
        res = np.zeros((n, nl), order="F")
        op_, ldo = res.ctypes.data, n
    else:
        if not _is_torch_cuda(out) or tuple(out.shape) != (n, nl) or (out.stride(0) != 1 and n > 1):
            raise ValueError("out must be a column-major float64 cuda tensor of shape (n, nlambda)")
        res, op_, ldo = out, out.data_ptr(), max(out.stride(1) if nl > 1 else n, n)
    if handle:
        _check(L.oemb200_predict_h(newx.handle, b.ctypes.data, rows, nl, 1 if response else 0, op_, ldo, ctypes.byref(o),
                                   ctypes.byref(st)))
    elif sparse:
        _check(L.oemb200_predict_sparse(rip, cpp, vp_, n, p, b.ctypes.data, rows, nl, 1 if response else 0, op_, ldo,
                                        ctypes.byref(o), ctypes.byref(st)))
    else:
        _check(L.oemb200_predict(xp, n, p, ld, b.ctypes.data, rows, nl, 1 if response else 0, op_, ldo, ctypes.byref(o),
                                 ctypes.byref(st)))
    return (res, st.as_dict()) if return_stats else res
