"""ctypes binding of libgpb200.so -- the same C ABI (include/gpb200.h) the Julia shim `ccall`s.

No CPU fallback: if the shared library is missing or no CUDA device is present, construction of an
`Engine` raises.  (The library is built in-tree by `__graft_entry__.build()` / `make -C csrc`.)
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libgpb200.so")

OK, EINVAL, ECUDA, ENCCL, ESTATE = 0, -1, -2, -3, -4

# opcodes (include/gpb200.h)
OP = dict(SE_ISO=1, SE_ARD=2, MAT12_ISO=3, MAT32_ISO=4, MAT52_ISO=5, MAT12_ARD=6, MAT32_ARD=7,
          MAT52_ARD=8, RQ_ISO=9, RQ_ARD=10, PERIODIC=11, LIN_ISO=12, LIN_ARD=13, POLY=14, NOISE=15,
          CONST=16, SUM=32, PROD=33)
MAX_OPS, MAX_THETA, MAX_DIMS, OP_STRIDE = 16, 96, 128, 6

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_H = C.c_void_p

_SIGNATURES = {
    "gpb200_create": (C.c_int, [C.POINTER(_H), C.c_int]),
    "gpb200_destroy": (None, [_H]),
    "gpb200_last_error": (C.c_char_p, [_H]),
    "gpb200_version": (C.c_int, []),
    "gpb200_set_data": (C.c_int, [_H, C.c_int64, C.c_int32, _dp, C.c_int64]),
    "gpb200_set_kernel": (C.c_int, [_H, C.c_int32, _ip, C.c_int32, _ip, C.c_int32]),
    "gpb200_factorize": (C.c_int, [_H, _dp, _dp, C.c_int64, C.c_double]),
    "gpb200_logdet": (C.c_int, [_H, _dp]),
    "gpb200_solve": (C.c_int, [_H, _dp, _dp]),
    "gpb200_mll": (C.c_int, [_H, _dp, _dp, _dp]),
    "gpb200_grad_prepare": (C.c_int, [_H]),
    "gpb200_grad_kernel": (C.c_int, [_H, _dp, _dp, _dp]),
    "gpb200_unwhiten": (C.c_int, [_H, _dp, _dp]),
    "gpb200_gpa_grad": (C.c_int, [_H, _dp, _dp, _dp, _dp]),
    "gpb200_get_chol_bar": (C.c_int, [_H, _dp]),
    "gpb200_predict": (C.c_int, [_H, C.c_int64, _dp, C.c_int64, _dp, _dp, _dp, _dp]),
    "gpb200_rand": (C.c_int, [_H, C.c_int64, _dp, C.c_int64, _dp, C.c_int64, _dp, C.c_double, _dp, _dp]),
    "gpb200_append": (C.c_int, [_H, C.c_int64, _dp, C.c_int64]),
    "gpb200_cv_param": (C.c_int, [_H, C.c_int32, _dp, _dp, _dp]),
    "gpb200_cv_block": (C.c_int, [_H, C.c_int32, C.c_int64, C.POINTER(C.c_int64), _dp]),
    "gpb200_get_gram": (C.c_int, [_H, _dp]),
    "gpb200_get_factor": (C.c_int, [_H, _dp]),
    "gpb200_get_inverse": (C.c_int, [_H, _dp]),
    "gpb200_get_inverse_diag": (C.c_int, [_H, _dp]),
    "gpb200_get_timings": (C.c_int, [_H, _dp, C.c_int32]),
    "gpb200_launch_count": (C.c_int64, [_H]),
    "gpb200_set_option": (C.c_int, [_H, C.c_char_p, C.c_int64]),
    "gpb200_set_stream": (C.c_int, [_H, C.c_void_p]),
    "gpb200_fp64_peak": (C.c_int, [_H, _dp, _dp]),
    "gpb200_dgemm_nt_device": (C.c_int, [_H, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_void_p,
                                         C.c_int64, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_int64,
                                         C.c_int, C.c_int, _dp]),
    "gpb200_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "gpb200_ipc_export": (C.c_int, [_H, C.c_void_p]),
    "gpb200_ipc_import": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "gpb200_fitc_create": (C.c_int, [C.POINTER(_H), C.c_int]),
    "gpb200_fitc_destroy": (None, [_H]),
    "gpb200_fitc_last_error": (C.c_char_p, [_H]),
    "gpb200_fitc_set_data": (C.c_int, [_H, C.c_int64, C.c_int32, _dp, C.c_int64, C.c_int64, _dp, C.c_int64]),
    "gpb200_fitc_set_kernel": (C.c_int, [_H, C.c_int32, _ip, C.c_int32, _ip, C.c_int32]),
    "gpb200_fitc_factorize": (C.c_int, [_H, _dp, C.c_double]),
    "gpb200_fitc_mll": (C.c_int, [_H, _dp, _dp, _dp, _dp]),
    "gpb200_fitc_grad_noise": (C.c_int, [_H, _dp]),
    "gpb200_fitc_grad_kernel": (C.c_int, [_H, _dp]),
    "gpb200_fitc_predict": (C.c_int, [_H, C.c_int64, _dp, C.c_int64, _dp, _dp]),
    "gpb200_fitc_comm_init": (C.c_int, [_H, C.c_int, C.c_int, C.c_char_p]),
    "gpb200_fitc_predict_cov": (C.c_int, [_H, C.c_int64, _dp, C.c_int64, _dp, _dp]),
    "gpb200_fitc_set_mode": (C.c_int, [_H, C.c_int]),
    "gpb200_fitc_launch_count": (C.c_int64, [_H]),
    "gpb200_comm_init": (C.c_int, [_H, C.c_int, C.c_int, C.c_char_p]),
    "gpb200_group_create": (C.c_int, [C.POINTER(_H), C.c_int]),
    "gpb200_storage_info": (C.c_int, [_H, C.POINTER(C.c_int64), C.c_int32]),
}

_lib = None


def declared_symbols():
    """Every symbol include/gpb200.h declares (used by the CPU-side ABI test)."""
    return sorted(_SIGNATURES)


def load_library():
    """dlopen libgpb200.so (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libgpb200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C gaussianprocesses.jl_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class PosDefException(np.linalg.LinAlgError):
    """Mirror of LinearAlgebra.PosDefException(info) thrown by cholesky! (src/GP.jl:110)."""

    def __init__(self, info):
        super().__init__("matrix is not positive definite; Cholesky factorization failed (leading minor %d)" % info)
        self.info = info


def _as_dp(a):
    return a.ctypes.data_as(_dp)


class Engine:
    """Owns one gpb200_handle (one GPU).  Thin, 1:1 with the C ABI."""

    def __init__(self, device=0):
        self._lib = load_library()
        self._h = _H()
        rc = self._lib.gpb200_create(C.byref(self._h), int(device))
        if rc != OK:
            msg = self._lib.gpb200_last_error(None)
            raise RuntimeError("gpb200_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.N = 0
        self.d = 0
        self.n_theta = 0

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.gpb200_destroy(self._h)
            self._h = _H()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc == OK:
            return
        msg = self._lib.gpb200_last_error(self._h)
        msg = msg.decode() if msg else ""
        if rc > 0:
            raise PosDefException(rc)
        if rc in (EINVAL, ESTATE):
            raise ValueError("%s: %s" % (what, msg))       # ArgumentError on the Julia side
        raise RuntimeError("%s failed (%d): %s" % (what, rc, msg))

    # -- data / model ---------------------------------------------------------------------
    def set_data(self, x_pm):
        """x_pm: (N, d) C-contiguous float64 == Julia's d x N column-major matrix."""
        x_pm = np.ascontiguousarray(x_pm, dtype=np.float64)
        N, d = x_pm.shape
        self._check(self._lib.gpb200_set_data(self._h, N, d, _as_dp(x_pm), d), "set_data")
        self.N, self.d = N, d

    def set_kernel(self, ops, dims, n_theta):
        ops = np.ascontiguousarray(ops, dtype=np.int32).reshape(-1, OP_STRIDE)
        dims = np.ascontiguousarray(dims, dtype=np.int32)
        self._check(self._lib.gpb200_set_kernel(self._h, ops.shape[0], ops.ctypes.data_as(_ip), dims.size,
                                                dims.ctypes.data_as(_ip), int(n_theta)), "set_kernel")
        self.n_theta = int(n_theta)

    def set_option(self, key, value):
        self._check(self._lib.gpb200_set_option(self._h, key.encode(), int(value)), "set_option")

    # -- hot path -------------------------------------------------------------------------
    def factorize(self, theta, log_noise, extra_nugget=0.0):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        ln = np.ascontiguousarray(np.atleast_1d(log_noise), dtype=np.float64)
        self._check(self._lib.gpb200_factorize(self._h, _as_dp(theta), _as_dp(ln), ln.size, float(extra_nugget)),
                    "factorize")

    def logdet(self):
        out = C.c_double()
        self._check(self._lib.gpb200_logdet(self._h, C.byref(out)), "logdet")
        return out.value

    def solve(self, rhs):
        rhs = np.ascontiguousarray(rhs, dtype=np.float64)
        if rhs.shape != (self.N,):
            raise ValueError("solve: rhs must have length N")
        out = np.empty(self.N)
        self._check(self._lib.gpb200_solve(self._h, _as_dp(rhs), _as_dp(out)), "solve")
        return out

    def mll(self, y_minus_mean):
        r = np.ascontiguousarray(y_minus_mean, dtype=np.float64)
        if r.shape != (self.N,):
            raise ValueError("mll: y must have length N")
        alpha = np.empty(self.N)
        out = C.c_double()
        self._check(self._lib.gpb200_mll(self._h, _as_dp(r), _as_dp(alpha), C.byref(out)), "mll")
        return alpha, out.value

    def grad_prepare(self):
        self._check(self._lib.gpb200_grad_prepare(self._h), "grad_prepare")

    def grad_kernel(self, alpha=None):
        g = np.empty(max(self.n_theta, 1))
        tr = C.c_double()
        ap = _as_dp(np.ascontiguousarray(alpha, dtype=np.float64)) if alpha is not None else None
        self._check(self._lib.gpb200_grad_kernel(self._h, ap, _as_dp(g), C.byref(tr)), "grad_kernel")
        return g[:self.n_theta].copy(), tr.value

    def unwhiten(self, v):
        """f = L v on the resident factor (GPA.jl:106)."""
        v = np.ascontiguousarray(v, dtype=np.float64)
        if v.shape != (self.N,):
            raise ValueError("unwhiten: v must have length N")
        f = np.empty(self.N)
        self._check(self._lib.gpb200_unwhiten(self._h, _as_dp(v), _as_dp(f)), "unwhiten")
        return f

    def gpa_grad(self, v, dl_df):
        """(L' dl_df, dll_kern) of the latent GP (GPA.jl:183-228); K^-1 and the resident alpha are gone afterwards."""
        v = np.ascontiguousarray(v, dtype=np.float64)
        g = np.ascontiguousarray(dl_df, dtype=np.float64)
        if v.shape != (self.N,) or g.shape != (self.N,):
            raise ValueError("gpa_grad: v and dl_df must have length N")
        dv = np.empty(self.N)
        dk = np.empty(max(self.n_theta, 1))
        self._check(self._lib.gpb200_gpa_grad(self._h, _as_dp(v), _as_dp(g), _as_dp(dv), _as_dp(dk)), "gpa_grad")
        return dv, dk[:self.n_theta].copy()

    def chol_bar(self):
        """debug: the symmetric P + P' of the last gpa_grad"""
        out = np.empty((self.N, self.N))
        self._check(self._lib.gpb200_get_chol_bar(self._h, _as_dp(out)), "get_chol_bar")
        return out

    def predict(self, xs_pm, alpha=None, want_var=True, full_cov=False):
        xs_pm = np.ascontiguousarray(xs_pm, dtype=np.float64)
        M, d = xs_pm.shape
        if d != self.d:
            raise ValueError("Gaussian Process object and input observations do not have consistent dimensions")
        mu = np.empty(M)
        var = np.empty(M) if want_var else None
        cov = np.empty((M, M)) if full_cov else None
        ap = _as_dp(np.ascontiguousarray(alpha, dtype=np.float64)) if alpha is not None else None
        self._check(self._lib.gpb200_predict(self._h, M, _as_dp(xs_pm), d, ap, _as_dp(mu),
                                             _as_dp(var) if want_var else None,
                                             _as_dp(cov) if full_cov else None), "predict")
        return mu, var, cov

    def rand(self, xs_pm, z, nugget=1e-10, alpha=None):
        """z: (nsamp, M) standard-normal draws (== Julia's M x nsamp column-major).  Returns (mu_minus_mean[M], samples (nsamp, M))."""
        xs_pm = np.ascontiguousarray(xs_pm, dtype=np.float64)
        z = np.ascontiguousarray(z, dtype=np.float64)
        M, d = xs_pm.shape
        if d != self.d or z.ndim != 2 or z.shape[1] != M:
            raise ValueError("rand: inconsistent dimensions")
        mu = np.empty(M)
        out = np.empty_like(z)
        ap = _as_dp(np.ascontiguousarray(alpha, dtype=np.float64)) if alpha is not None else None
        self._check(self._lib.gpb200_rand(self._h, M, _as_dp(xs_pm), d, ap, z.shape[0], _as_dp(z), float(nugget), _as_dp(mu),
                                          _as_dp(out)), "rand")
        return mu, out

    def append(self, xnew_pm):
        """extend the factor by the rows of xnew_pm (k, d) with unchanged hyper-parameters (ElasticGPE append!)"""
        xnew_pm = np.ascontiguousarray(xnew_pm, dtype=np.float64)
        k, d = xnew_pm.shape
        if d != self.d:
            raise ValueError("append: wrong input dimension")
        self._check(self._lib.gpb200_append(self._h, k, _as_dp(xnew_pm), d), "append")
        self.N += k

    def cv_param(self, param, alpha=None):
        """(Z_j alpha, diag(Z_j K^-1)) for kernel parameter `param` (index into the full parameter vector) or -1 = noise."""
        za, dg = np.empty(self.N), np.empty(self.N)
        ap = _as_dp(np.ascontiguousarray(alpha, dtype=np.float64)) if alpha is not None else None
        self._check(self._lib.gpb200_cv_param(self._h, int(param), ap, _as_dp(za), _as_dp(dg)), "cv_param")
        return za, dg

    def cv_block(self, which, idx):
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        out = np.empty((idx.size, idx.size))
        self._check(self._lib.gpb200_cv_block(self._h, int(which), idx.size, idx.ctypes.data_as(C.POINTER(C.c_int64)), _as_dp(out)), "cv_block")
        return out

    # -- debug ----------------------------------------------------------------------------
    def gram(self):
        K = np.empty((self.N, self.N))
        self._check(self._lib.gpb200_get_gram(self._h, _as_dp(K)), "get_gram")
        return K

    def factor_upper(self):
        """U (upper) with K_y = U'U, as a numpy (N, N) array (row i, col j -> U[i, j])."""
        buf = np.empty((self.N, self.N))
        self._check(self._lib.gpb200_get_factor(self._h, _as_dp(buf)), "get_factor")
        return buf.T.copy()      # buffer is column-major U == row-major L

    def inverse(self):
        K = np.empty((self.N, self.N))
        self._check(self._lib.gpb200_get_inverse(self._h, _as_dp(K)), "get_inverse")
        return K

    def inverse_diag(self):
        d = np.empty(self.N)
        self._check(self._lib.gpb200_get_inverse_diag(self._h, _as_dp(d)), "get_inverse_diag")
        return d

    def storage_info(self):
        v = (C.c_int64 * 8)()
        self._check(self._lib.gpb200_storage_info(self._h, v, 8), "storage_info")
        return dict(sharded=bool(v[0]), bytes_F=int(v[1]), bytes_G=int(v[2]), rb=int(v[3]), nranks=int(v[4]), rank=int(v[5]),
                    tma=bool(v[6]))

    def _own_rows_inverse(self):
        """sharded storage: this rank's rows of K^-1 (lower part valid), zeros elsewhere"""
        K = np.empty((self.N, self.N))
        self._check(self._lib.gpb200_get_inverse(self._h, _as_dp(K)), "get_inverse")
        return np.tril(K)

    def timings(self):
        ms = np.zeros(16)
        self._check(self._lib.gpb200_get_timings(self._h, _as_dp(ms), 16), "get_timings")
        return dict(gram=ms[0], cholesky=ms[1], solve_mll=ms[2], inverse=ms[3], trace=ms[4], predict=ms[5],
                    gemm_launches=ms[6], gemm_ms=ms[7], gemm_flops=ms[8], gpa_unwhiten=ms[9], gpa_trmv_t=ms[10],
                    gpa_merges=ms[11], gpa_scan=ms[12], gpa_gemms=ms[13])

    def set_stream(self, cuda_stream):
        """Run on the caller's CUDA stream (int handle, e.g. torch.cuda.current_stream().cuda_stream); 0/None = private."""
        self._check(self._lib.gpb200_set_stream(self._h, C.c_void_p(int(cuda_stream) if cuda_stream else None)), "set_stream")

    # -- multi-GPU (one process per GPU) -------------------------------------------------------
    def nccl_unique_id(self):
        buf = C.create_string_buffer(128)
        rc = (self._lib if self is not None else load_library()).gpb200_nccl_unique_id(C.cast(buf, C.c_void_p))
        if rc != OK:
            raise RuntimeError("gpb200_nccl_unique_id failed (%d)" % rc)
        return buf.raw

    def comm_init(self, nranks, rank, id128):
        if len(id128) != 128:
            raise ValueError("NCCL unique id must be 128 bytes")
        ib = C.create_string_buffer(bytes(id128), 128)
        self._check(self._lib.gpb200_comm_init(self._h, int(nranks), int(rank), C.cast(ib, C.c_char_p)), "comm_init")
        self.nranks, self.rank = int(nranks), int(rank)

    IPC_BYTES = 512

    def ipc_export(self):
        buf = C.create_string_buffer(self.IPC_BYTES)
        self._check(self._lib.gpb200_ipc_export(self._h, C.cast(buf, C.c_void_p)), "ipc_export")
        return buf.raw

    def ipc_import(self, blobs):
        """blobs: list of nranks byte strings in rank order (own entry ignored)."""
        joined = b"".join(bytes(b) for b in blobs)
        if len(joined) != self.IPC_BYTES * len(blobs):
            raise ValueError("ipc_import: every blob must be %d bytes" % self.IPC_BYTES)
        buf = C.create_string_buffer(joined, len(joined))
        self._check(self._lib.gpb200_ipc_import(self._h, len(blobs), C.cast(buf, C.c_void_p)), "ipc_import")

    def fp64_peak(self):
        a, b = C.c_double(), C.c_double()
        self._check(self._lib.gpb200_fp64_peak(self._h, C.byref(a), C.byref(b)), "fp64_peak")
        return dict(dmma_tflops=a.value, dfma_tflops=b.value)

    def launch_count(self):
        return int(self._lib.gpb200_launch_count(self._h))

    def dgemm_nt_device(self, impl, M, N, K, alpha, dA, lda, dB, ldb, beta, dC, ldc, lower_only=False, reps=1):
        ms = C.c_double()
        self._check(self._lib.gpb200_dgemm_nt_device(self._h, int(impl), M, N, K, float(alpha), C.c_void_p(dA), lda,
                                                     C.c_void_p(dB), ldb, float(beta), C.c_void_p(dC), ldc,
                                                     1 if lower_only else 0, int(reps), C.byref(ms)), "dgemm_nt")
        return ms.value


class FitcEngine:
    """Owns one gpb200_fitc handle: the FITC sparse strategy (src/sparse/fully_indep_train_conditional.jl)."""

    def __init__(self, device=0):
        self._lib = load_library()
        self._h = _H()
        rc = self._lib.gpb200_fitc_create(C.byref(self._h), int(device))
        if rc != OK:
            msg = self._lib.gpb200_last_error(None)
            raise RuntimeError("gpb200_fitc_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.N = self.M = self.d = 0

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.gpb200_fitc_destroy(self._h)
            self._h = _H()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc == OK:
            return
        msg = self._lib.gpb200_fitc_last_error(self._h)
        msg = msg.decode() if msg else ""
        if rc > 0:
            raise PosDefException(rc)
        if rc in (EINVAL, ESTATE):
            raise ValueError("%s: %s" % (what, msg))
        raise RuntimeError("%s failed (%d): %s" % (what, rc, msg))

    def set_data(self, x_pm, xu_pm):
        x_pm = np.ascontiguousarray(x_pm, dtype=np.float64)
        xu_pm = np.ascontiguousarray(xu_pm, dtype=np.float64)
        (N, d), (M, d2) = x_pm.shape, xu_pm.shape
        if d != d2:
            raise ValueError("inducing points and inputs must have the same dimension")
        self._check(self._lib.gpb200_fitc_set_data(self._h, N, d, _as_dp(x_pm), d, M, _as_dp(xu_pm), d), "fitc_set_data")
        self.N, self.M, self.d = N, M, d

    def grad_kernel(self):
        g = np.empty(max(self.n_theta, 1))
        self._check(self._lib.gpb200_fitc_grad_kernel(self._h, _as_dp(g)), "fitc_grad_kernel")
        return g[:self.n_theta].copy()

    def set_kernel(self, ops, dims, n_theta):
        self.n_theta = int(n_theta)
        ops = np.ascontiguousarray(ops, dtype=np.int32).reshape(-1, OP_STRIDE)
        dims = np.ascontiguousarray(dims, dtype=np.int32)
        self._check(self._lib.gpb200_fitc_set_kernel(self._h, ops.shape[0], ops.ctypes.data_as(_ip), dims.size,
                                                     dims.ctypes.data_as(_ip), int(n_theta)), "fitc_set_kernel")

    def factorize(self, theta, log_noise):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        self._check(self._lib.gpb200_fitc_factorize(self._h, _as_dp(theta), float(log_noise)), "fitc_factorize")

    def mll(self, y_minus_mean):
        r = np.ascontiguousarray(y_minus_mean, dtype=np.float64)
        if r.shape != (self.N,):
            raise ValueError("fitc_mll: y must have length N")
        alpha = np.empty(self.N)
        m, ld = C.c_double(), C.c_double()
        self._check(self._lib.gpb200_fitc_mll(self._h, _as_dp(r), _as_dp(alpha), C.byref(m), C.byref(ld)), "fitc_mll")
        return alpha, m.value, ld.value

    def grad_noise(self):
        g = C.c_double()
        self._check(self._lib.gpb200_fitc_grad_noise(self._h, C.byref(g)), "fitc_grad_noise")
        return g.value

    def predict(self, xs_pm, want_var=True):
        xs_pm = np.ascontiguousarray(xs_pm, dtype=np.float64)
        Ms, d = xs_pm.shape
        if d != self.d:
            raise ValueError("Gaussian Process object and input observations do not have consistent dimensions")
        mu = np.empty(Ms)
        var = np.empty(Ms) if want_var else None
        self._check(self._lib.gpb200_fitc_predict(self._h, Ms, _as_dp(xs_pm), d, _as_dp(mu),
                                                  _as_dp(var) if want_var else None), "fitc_predict")
        return mu, var

    def comm_init(self, nranks, rank, id128):
        ib = C.create_string_buffer(bytes(id128), 128)
        self._check(self._lib.gpb200_fitc_comm_init(self._h, int(nranks), int(rank), C.cast(ib, C.c_char_p)), "fitc_comm_init")

    def predict_cov(self, xs_pm):
        xs_pm = np.ascontiguousarray(xs_pm, dtype=np.float64)
        Ms, d = xs_pm.shape
        if d != self.d:
            raise ValueError("Gaussian Process object and input observations do not have consistent dimensions")
        mu = np.empty(Ms)
        cov = np.empty((Ms, Ms))
        self._check(self._lib.gpb200_fitc_predict_cov(self._h, Ms, _as_dp(xs_pm), d, _as_dp(mu), _as_dp(cov)), "fitc_predict_cov")
        return mu, cov

    def set_mode(self, mode):
        """0 FITC, 1 DTC, 2 SoR."""
        self._check(self._lib.gpb200_fitc_set_mode(self._h, int(mode)), "fitc_set_mode")

    def launch_count(self):
        return int(self._lib.gpb200_fitc_launch_count(self._h))


class LocalGroupEngine:
    """R engines on ONE device acting as the R ranks of the ROW-SHARDED multi-GPU schedules (gpb200_group_create,
    csrc/shard_impl.cuh): each virtual rank maps only its own block rows of the N x N factor / inverse, collectives are
    event-ordered device copies.  Same interface as `Engine`, so `GPE(..., engine=LocalGroupEngine(4))` runs the whole
    host mirror over the sharded storage on a single GPU (tests; the production path is one process per GPU + NCCL)."""

    def __init__(self, nranks, device=0, rb=0):
        self.engines = [Engine(device) for _ in range(int(nranks))]
        self.lead = self.engines[0]
        arr = (_H * len(self.engines))(*[e._h for e in self.engines])
        rc = self.lead._lib.gpb200_group_create(arr, len(self.engines))
        self.lead._check(rc, "group_create")
        self.nranks = len(self.engines)
        if rb:
            self.set_option("shard_rb", rb)

    # replicated state: every virtual rank gets it
    def set_data(self, x_pm):
        for e in self.engines:
            e.set_data(x_pm)
        self.N, self.d = self.lead.N, self.lead.d

    def set_kernel(self, ops, dims, n_theta):
        for e in self.engines:
            e.set_kernel(ops, dims, n_theta)
        self.n_theta = self.lead.n_theta

    def set_option(self, key, value):
        for e in self.engines:
            e.set_option(key, value)

    def close(self):
        for e in self.engines:
            e.close()

    # collective entry points: the leader drives every rank
    def factorize(self, *a, **k):
        return self.lead.factorize(*a, **k)

    def mll(self, *a, **k):
        return self.lead.mll(*a, **k)

    def solve(self, *a, **k):
        return self.lead.solve(*a, **k)

    def logdet(self):
        return self.lead.logdet()

    def grad_prepare(self):
        return self.lead.grad_prepare()

    def grad_kernel(self, *a, **k):
        return self.lead.grad_kernel(*a, **k)

    def predict(self, *a, **k):
        return self.lead.predict(*a, **k)

    def unwhiten(self, *a, **k):
        return self.lead.unwhiten(*a, **k)

    def gpa_grad(self, *a, **k):
        return self.lead.gpa_grad(*a, **k)

    def rand(self, *a, **k):
        return self.lead.rand(*a, **k)

    def timings(self):
        return self.lead.timings()

    def launch_count(self):
        return sum(e.launch_count() for e in self.engines)

    def gram(self):
        return self.lead.gram()

    # debug getters: every rank returns its own rows (zeros elsewhere); the pieces add up to the full matrix
    def factor_upper(self):
        return sum(e.factor_upper() for e in self.engines)

    def inverse(self):
        K = sum(e._own_rows_inverse() for e in self.engines)
        return np.tril(K) + np.tril(K, -1).T

    def inverse_diag(self):
        return np.diag(self.inverse()).copy()
