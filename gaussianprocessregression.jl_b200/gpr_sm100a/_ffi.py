"""ctypes binding of libgpr_sm100a.so (include/gpr_sm100a.h).

This is the executed stand-in for the Julia `ccall` glue (julia/GPRsm100a.jl):
same entry points, same argument meaning.  There is no fallback: if the shared
library or a usable sm_100 device is missing, importing works but the first call
raises.
"""
import ctypes as C
import os
import re

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
ROOT = os.path.dirname(PKG)
LIB_PATH = os.path.join(PKG, "libgpr_sm100a.so")
HEADER = os.path.join(ROOT, "include", "gpr_sm100a.h")

GPR_OK = 0
GPR_ERR_NOT_POSDEF = 1
KERN_SE, KERN_NOISE, KERN_MATERN52 = 1, 2, 3
FETCH_U, FETCH_ALPHA, FETCH_KINV, FETCH_WT = 0, 1, 2, 3
T_NAMES = ["kbuild", "potrf", "potrs", "trtri", "lauum", "grad", "total", "pred_kstar", "pred_mean", "pred_trsm",
           "pred_rownorm", "eval", "split_build", "split_gemm", "split_d2h"]
T_COUNT = 16

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_i64 = C.c_int64
_vp = C.c_void_p

_SIGS = {
    "gpr_version": (C.c_int, []),
    "gpr_device_count": (C.c_int, []),
    "gpr_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "gpr_ctx_destroy": (C.c_int, [_vp]),
    "gpr_last_error": (C.c_char_p, [_vp]),
    "gpr_ctx_set_option": (C.c_int, [_vp, C.c_char_p, _i64]),
    "gpr_dbg_ozaki_dgemm": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, _dp, _i64, _dp, _i64, C.c_double, _dp, _i64,
                                      C.c_int, C.c_int, _dp]),
    "gpr_ctx_launch_count": (_i64, [_vp]),
    "gpr_dim_hp": (C.c_int, [_ip, C.c_int, C.c_int]),
    "gpr_model_create": (C.c_int, [_vp, _ip, C.c_int, C.c_int, _i64, _dp, _dp, C.c_int, C.c_int, C.POINTER(_vp)]),
    "gpr_model_destroy": (C.c_int, [_vp]),
    "gpr_model_set_y": (C.c_int, [_vp, _dp]),
    "gpr_model_set_x": (C.c_int, [_vp, _dp]),
    "gpr_kernel": (C.c_int, [_vp, _ip, C.c_int, C.c_int, _dp, _dp, _i64, _dp, _i64, C.c_int, C.c_double, C.c_int, _dp]),
    "gpr_kernel_grad": (C.c_int, [_vp, C.c_int, C.c_int, _dp, _dp, _i64, C.c_int, C.c_double, _dp]),
    "gpr_update_cache": (C.c_int, [_vp, _dp, C.c_int, C.c_double, C.c_int, C.POINTER(_i64)]),
    "gpr_loss": (C.c_int, [_vp, _dp]),
    "gpr_grad": (C.c_int, [_vp, C.c_int, _dp]),
    "gpr_nlml_grad": (C.c_int, [_vp, _dp, C.c_int, C.c_int, C.c_double, _dp, _dp, C.POINTER(_i64)]),
    "gpr_fetch": (C.c_int, [_vp, C.c_int, _dp]),
    "gpr_predict": (C.c_int, [_vp, _dp, _i64, C.c_int, _dp, _dp, _dp]),
    "gpr_predict_device": (C.c_int, [_vp, _vp, _i64, C.c_int, _vp, _vp]),
    "gpr_split_kernel": (C.c_int, [_vp, _ip, C.c_int, C.c_int, _dp, _dp, _i64, _dp, _i64, _dp, _i64, _dp, _dp, _dp]),
    "gpr_split_predict": (C.c_int, [_vp, _dp, _i64, _dp, _i64, _i64, _i64, _dp, _dp]),
    "gpr_timings": (C.c_int, [_vp, _dp, C.c_int]),
    "gpr_model_route": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "gpr_integrate": (C.c_int, [_vp, _dp, _dp, _dp, _dp]),
    "gpr_integrate_batch": (C.c_int, [_vp, _i64, _dp, _dp, _dp, _dp]),
    "gpr_sample_mvn": (C.c_int, [_vp, _ip, C.c_int, C.c_int, _dp, _dp, _i64, C.c_double, _dp, _dp, _dp, C.POINTER(_i64)]),
    "gpr_dbg_dgemm": (C.c_int, [_vp, C.c_char, C.c_char, C.c_int, C.c_int, C.c_int, C.c_double, _dp, _i64, _dp, _i64,
                                C.c_double, _dp, _i64, C.c_int, C.c_int, _dp]),
    "gpr_dbg_factor": (C.c_int, [_vp, _dp, _i64, C.c_int, C.POINTER(_i64), _dp]),
    "gpr_mgpu_create": (C.c_int, [C.c_int, _ip, _i64, C.POINTER(_vp)]),
    "gpr_dist_unique_id": (C.c_int, [_vp]),
    "gpr_dist_create": (C.c_int, [C.c_int, C.c_int, C.c_int, _vp, _i64, C.POINTER(_vp)]),
    "gpr_mgpu_destroy": (C.c_int, [_vp]),
    "gpr_mgpu_set_option": (C.c_int, [_vp, C.c_char_p, _i64]),
    "gpr_mgpu_last_error": (C.c_char_p, [_vp]),
    "gpr_mgpu_launch_count": (_i64, [_vp]),
    "gpr_mgpu_model_create": (C.c_int, [_vp, _ip, C.c_int, C.c_int, _i64, _dp, _dp, C.c_int, C.c_int, C.POINTER(_vp)]),
    "gpr_mgpu_model_destroy": (C.c_int, [_vp]),
    "gpr_mgpu_nlml_grad": (C.c_int, [_vp, _dp, C.c_int, C.c_int, C.c_double, _dp, _dp, C.POINTER(_i64)]),
    "gpr_mgpu_update_cache": (C.c_int, [_vp, _dp, C.c_int, C.c_double, C.POINTER(_i64)]),
    "gpr_mgpu_predict": (C.c_int, [_vp, _dp, _i64, C.c_int, _dp, _dp, _dp]),
    "gpr_mgpu_split_predict": (C.c_int, [_vp, _dp, _i64, _dp, _i64, _i64, _i64, _dp, _dp]),
    "gpr_mgpu_integrate": (C.c_int, [_vp, _i64, _dp, _dp, _dp, _dp]),
    "gpr_mgpu_fetch": (C.c_int, [_vp, C.c_int, _dp]),
    "gpr_mgpu_timings": (C.c_int, [_vp, _dp, C.c_int]),
    "gpr_mgpu_dbg_factor": (C.c_int, [_vp, _dp, _i64, _dp, C.c_int, C.c_int, C.POINTER(_i64), _dp]),
}


def header_symbols():
    """Every function name declared in include/gpr_sm100a.h."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gpr_[a-z0-9_]+)\s*\(", text)))


_lib = None


def lib():
    """Load the shared library (no device needed for loading)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python gaussianprocessregression.jl_b200/build.py` "
                "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def device_count():
    """Number of usable sm_100-class devices (0 when there is none: nothing in this package runs then)."""
    return int(lib().gpr_device_count())


class GPRError(RuntimeError):
    pass


class PosDefException(GPRError):
    """Mirror of Julia's PosDefException thrown by cholesky!(...; check=true) (src/cost.jl:77)."""

    def __init__(self, info):
        super().__init__(f"matrix is not positive definite; Cholesky factorization failed (info = {info}).")
        self.info = info


def dptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def f64(a, order="F"):
    """float64 array in column-major (Julia) storage; copies only when needed."""
    return np.require(a, dtype=np.float64, requirements=["F_CONTIGUOUS", "ALIGNED"] if order == "F" else ["C_CONTIGUOUS", "ALIGNED"])


def types_array(types):
    arr = (C.c_int * len(types))(*types)
    return arr


class Context:
    """One library context (= one GPU, one stream)."""

    def __init__(self, device=0):
        self._h = _vp()
        rc = lib().gpr_ctx_create(int(device), C.byref(self._h))
        if rc != 0:
            msg = lib().gpr_last_error(None)
            self._h = None
            raise GPRError(f"gpr_ctx_create(device={device}) failed ({rc}): {msg.decode() if msg else ''}")
        self.device = device

    def check(self, rc, info=None):
        if rc == 0:
            return
        if rc == GPR_ERR_NOT_POSDEF:
            raise PosDefException(int(info.value) if info is not None else -1)
        msg = lib().gpr_last_error(self._h)
        raise GPRError(f"libgpr_sm100a error {rc}: {msg.decode() if msg else ''}")

    @property
    def handle(self):
        if self._h is None:
            raise GPRError("context destroyed")
        return self._h

    def set_option(self, name, value):
        self.check(lib().gpr_ctx_set_option(self.handle, name.encode(), int(value)))

    def launch_count(self):
        return int(lib().gpr_ctx_launch_count(self.handle))

    def close(self):
        if self._h is not None:
            lib().gpr_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def get_context(device=None):
    """Process-wide default context for a device (LOCAL_RANK under torchrun, else 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


class ModelHandle:
    """gpr_model: device-resident x, y, factor, weights, inverse for one GPRModel."""

    def __init__(self, ctx, types, D, x, y, train_axis=1):
        self.ctx = ctx
        self.types = list(types)
        x = f64(x)
        y2 = f64(y.reshape(y.shape[0], -1))
        self.D, self.N = int(x.shape[0]), int(x.shape[1])
        self.ny = int(y2.shape[1])
        if D != self.D:
            raise GPRError("x dimension mismatch")
        if y2.shape[0] != self.N:
            raise GPRError("x and y size mismatch.")
        self.P = lib().gpr_dim_hp(types_array(self.types), len(self.types), self.D)
        self._h = _vp()
        rc = lib().gpr_model_create(ctx.handle, types_array(self.types), len(self.types), self.D, self.N, dptr(x), dptr(y2),
                                    self.ny, int(train_axis), C.byref(self._h))
        if rc != 0:
            self._h = None
        ctx.check(rc)

    @property
    def handle(self):
        if self._h is None:
            raise GPRError("model destroyed")
        return self._h

    def set_y(self, y):
        y2 = f64(y.reshape(y.shape[0], -1))
        self.ctx.check(lib().gpr_model_set_y(self.handle, dptr(y2)))

    def set_x(self, x):
        self.ctx.check(lib().gpr_model_set_x(self.handle, dptr(f64(x))))

    def update_cache(self, hp, eps=1e-8, want_inverse=False):
        hp = f64(np.asarray(hp, dtype=np.float64).ravel())
        info = _i64(0)
        rc = lib().gpr_update_cache(self.handle, dptr(hp), hp.size, float(eps), int(bool(want_inverse)), C.byref(info))
        self.ctx.check(rc, info)

    def loss(self):
        F = C.c_double(0.0)
        self.ctx.check(lib().gpr_loss(self.handle, C.byref(F)))
        return F.value

    def grad(self, log_scale=False):
        G = np.empty(self.P)
        self.ctx.check(lib().gpr_grad(self.handle, int(bool(log_scale)), dptr(G)))
        return G

    def nlml_grad(self, hp, log_scale=False, eps=1e-8, want_f=True, want_g=True):
        hp = f64(np.asarray(hp, dtype=np.float64).ravel())
        F = C.c_double(0.0)
        G = np.empty(self.P) if want_g else None
        info = _i64(0)
        rc = lib().gpr_nlml_grad(self.handle, dptr(hp), hp.size, int(bool(log_scale)), float(eps),
                                 C.byref(F) if want_f else None, dptr(G), C.byref(info))
        self.ctx.check(rc, info)
        return (F.value if want_f else None), G

    def fetch(self, which):
        N = self.N
        if which in (FETCH_U, FETCH_KINV):
            out = np.empty((N, N), order="F")
        elif which == FETCH_ALPHA:
            out = np.empty(N)
        else:
            out = np.empty((N, self.ny), order="F")
        self.ctx.check(lib().gpr_fetch(self.handle, which, dptr(out)))
        return out

    def predict(self, xp, same_x=False, want_var=False, want_cov=False):
        xp = f64(xp)
        M = int(xp.shape[1])
        mean = np.empty((M, self.ny), order="F")
        var = np.empty(M) if want_var else None
        cov = np.empty((M, M), order="F") if want_cov else None
        self.ctx.check(lib().gpr_predict(self.handle, dptr(xp), M, int(bool(same_x)), dptr(mean), dptr(var), dptr(cov)))
        return mean, var, cov

    def predict_device(self, d_xp_ptr, M, d_mean_ptr, d_var_ptr=None, same_x=False):
        self.ctx.check(lib().gpr_predict_device(self.handle, _vp(d_xp_ptr), int(M), int(bool(same_x)), _vp(d_mean_ptr),
                                                _vp(d_var_ptr) if d_var_ptr else None))

    def split_predict(self, xe, xq, var_range=None, want_var=True, mean_out=None, var_out=None):
        """mean_out / var_out: caller-owned result arrays (the reference's predict!(mu, Sigma, ...) writes in place too); a fresh
        134 MB array per call costs more in first-touch page faults under the device-to-host copy than the whole computation."""
        xe, ne, xq, nq, lo, hi, mean, var = _split_args(xe, xq, var_range, want_var, mean_out, var_out)
        self.ctx.check(lib().gpr_split_predict(self.handle, dptr(xe), ne, dptr(xq), nq, lo, hi, dptr(mean), dptr(var)))
        return mean, var

    def integrate(self, a, b, want_var=True):
        """a, b of shape (D,): gpr_integrate, (Iout (ny,), var (1,)); of shape (D, nbox): gpr_integrate_batch,
        (Iout (nbox, ny), var (nbox,)), one triangular solve per tile of boxes."""
        a, b, nbox, single = _box_args(a, b, self.D)
        var = np.empty(nbox) if want_var else None
        if single:
            Iout = np.empty(self.ny)
            self.ctx.check(lib().gpr_integrate(self.handle, dptr(a), dptr(b), dptr(Iout), dptr(var)))
            return Iout, var
        Iout = np.empty((nbox, self.ny), order="F")
        self.ctx.check(lib().gpr_integrate_batch(self.handle, nbox, dptr(a), dptr(b), dptr(Iout), dptr(var)))
        return Iout, var

    def route(self):
        """(digits, digits_inverse) of the INT8-tensor-core route the last factorization took; 0 = FP64 DMMA pipe."""
        a, b = C.c_int(0), C.c_int(0)
        self.ctx.check(lib().gpr_model_route(self.handle, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def timings(self):
        ms = np.zeros(T_COUNT)
        self.ctx.check(lib().gpr_timings(self.handle, dptr(ms), T_COUNT))
        return {n: float(ms[i]) for i, n in enumerate(T_NAMES)}

    def close(self):
        if self._h is not None:
            lib().gpr_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _box_args(a, b, D):
    """(a, b, nbox, single) of the integrate entry points: bounds of shape (D,) (one box) or (D, nbox), the same for a and b,
    as D x nbox column-major arrays"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape or a.ndim not in (1, 2) or a.shape[0] != D or a.ndim == 2 and a.shape[1] < 1:
        raise GPRError("integration bounds must be (D,) or (D, nbox) arrays of the same shape")
    single, nbox = a.ndim == 1, 1 if a.ndim == 1 else int(a.shape[1])
    return f64(a.reshape(D, nbox)), f64(b.reshape(D, nbox)), nbox, single


def _split_args(xe, xq, var_range, want_var, mean_out, var_out):
    """(xe, ne, xq, nq, e_lo, e_hi, mean, var) of gpr_split_predict / gpr_mgpu_split_predict; mean and var are the caller's
    arrays when given (checked), fresh ones otherwise (var None unless want_var)."""
    xe, xq = f64(xe), f64(xq)
    ne, nq = int(xe.shape[1]), int(xq.shape[1])
    if mean_out is not None and (mean_out.shape != (ne, nq) or mean_out.dtype != np.float64 or not mean_out.flags.f_contiguous):
        raise GPRError("mean_out must be a Fortran-ordered float64 array of shape (ne, nq)")
    if var_out is not None and (var_out.shape != (ne * nq,) or var_out.dtype != np.float64 or not var_out.flags.c_contiguous):
        raise GPRError("var_out must be a contiguous float64 vector of length ne * nq")
    mean = mean_out if mean_out is not None else np.empty((ne, nq), order="F")
    var = (var_out if var_out is not None else np.empty(ne * nq)) if want_var else None
    lo, hi = (1, 0) if var_range is None else (int(var_range[0]), int(var_range[1]))
    return xe, ne, xq, nq, lo, hi, mean, var


def kernel_matrix(ctx, types, D, hp, x, xp, same_x, eps, add_noise):
    x = f64(x)
    xp = x if same_x else f64(xp)
    hp = f64(np.asarray(hp, dtype=np.float64).ravel())
    N, M = int(x.shape[1]), int(xp.shape[1])
    out = np.empty((N, M), order="F")
    ctx.check(lib().gpr_kernel(ctx.handle, types_array(types), len(types), int(D), dptr(hp), dptr(x), N, dptr(xp), M,
                               int(bool(same_x)), float(eps), int(bool(add_noise)), dptr(out)))
    return out


def kernel_grad_matrix(ctx, comp_type, D, hp_comp, x, li, eps):
    x = f64(x)
    hp_comp = f64(np.asarray(hp_comp, dtype=np.float64).ravel())
    N = int(x.shape[1])
    out = np.empty((N, N), order="F")
    ctx.check(lib().gpr_kernel_grad(ctx.handle, int(comp_type), int(D), dptr(hp_comp), dptr(x), N, int(li), float(eps), dptr(out)))
    return out


def split_kernel_arrays(ctx, types, D, hp, xe, xq, x):
    xe, xq, x = f64(xe), f64(xq), f64(x)
    hp = f64(np.asarray(hp, dtype=np.float64).ravel())
    ne, nq, N = int(xe.shape[1]), int(xq.shape[1]), int(x.shape[1])
    nk = sum(1 for t in types if t != KERN_NOISE)
    A = np.empty((ne, nq, nk), order="F")
    B = np.empty((ne, N, nk), order="F")
    Cc = np.empty((N, nq, nk), order="F")
    ctx.check(lib().gpr_split_kernel(ctx.handle, types_array(types), len(types), int(D), dptr(hp), dptr(xe), ne, dptr(xq), nq,
                                     dptr(x), N, dptr(A), dptr(B), dptr(Cc)))
    return A, B, Cc


def sample_mvn(ctx, types, D, hp, x, z, mu=None, shift=1e-7):
    """out = chol(kernel(cov, hp, x) .+ shift).L @ z + mu  (src/distributions.jl:20-45)"""
    x = f64(x)
    hp = f64(np.asarray(hp, dtype=np.float64).ravel())
    z = f64(np.asarray(z, dtype=np.float64).ravel())
    N = int(x.shape[1])
    if z.size != N:
        raise GPRError("z must hold one standard-normal draw per point")
    mu_c = None if mu is None else f64(np.asarray(mu, dtype=np.float64).ravel())
    out = np.empty(N)
    info = _i64(0)
    rc = lib().gpr_sample_mvn(ctx.handle, types_array(types), len(types), int(D), dptr(hp), dptr(x), N, float(shift), dptr(z),
                              dptr(mu_c), dptr(out), C.byref(info))
    ctx.check(rc, info)
    return out


def dbg_dgemm(ctx, transA, transB, alpha, A, B, beta, Cm, flags=0, reps=1):
    A, B = f64(A), f64(B)
    Cm = np.array(Cm, dtype=np.float64, order="F")
    M, N = Cm.shape
    K = A.shape[0] if transA == "T" else A.shape[1]
    ms = C.c_double(0.0)
    ctx.check(lib().gpr_dbg_dgemm(ctx.handle, transA.encode(), transB.encode(), M, N, K, float(alpha), dptr(A), A.shape[0],
                                  dptr(B), B.shape[0], float(beta), dptr(Cm), Cm.shape[0], int(flags), int(reps), C.byref(ms)))
    return Cm, ms.value


def dbg_ozaki_dgemm(ctx, alpha, A, B, beta, Cm, S=8, flags=0, reps=1):
    """C = alpha A^T B + beta C through the INT8 tensor cores (csrc/ozaki_i8.cuh).  A: (K, M), B: (K, N), Fortran ordered."""
    A, B = f64(A), f64(B)
    Cm = np.array(Cm, dtype=np.float64, order="F")
    K, M = A.shape
    N = B.shape[1]
    ms = C.c_double(0.0)
    ctx.check(lib().gpr_dbg_ozaki_dgemm(ctx.handle, M, N, K, int(S), float(alpha), dptr(A), A.shape[0], dptr(B), B.shape[0], float(beta),
                                        dptr(Cm), Cm.shape[0], int(flags), int(reps), C.byref(ms)))
    return Cm, ms.value


def dbg_factor(ctx, A, mode=0):
    A = np.array(A, dtype=np.float64, order="F")
    info = _i64(0)
    ms = C.c_double(0.0)
    rc = lib().gpr_dbg_factor(ctx.handle, dptr(A), A.shape[0], int(mode), C.byref(info), C.byref(ms))
    ctx.check(rc, info)
    return A, ms.value


class MultiContext:
    """gpr_mgpu: one process driving several ranks (one per entry of `devices`; a device may repeat) for the
    block-cyclic multi-GPU NLML + gradient (BASELINE.json config 5)."""

    def __init__(self, devices, nb=1024, transport=0):
        self.devices = [int(d) for d in devices]
        self.nb = int(nb)
        self._h = _vp()
        arr = (C.c_int * len(self.devices))(*self.devices)
        rc = lib().gpr_mgpu_create(len(self.devices), arr, self.nb, C.byref(self._h))
        if rc != 0:
            msg = lib().gpr_mgpu_last_error(None)
            self._h = None
            raise GPRError(f"gpr_mgpu_create(devices={self.devices}) failed ({rc}): {msg.decode() if msg else ''}")
        if transport:
            self.set_option("transport", transport)

    @property
    def handle(self):
        if self._h is None:
            raise GPRError("multi-GPU context destroyed")
        return self._h

    def check(self, rc, info=None):
        if rc == 0:
            return
        if rc == GPR_ERR_NOT_POSDEF:
            raise PosDefException(int(info.value) if info is not None else -1)
        msg = lib().gpr_mgpu_last_error(self._h)
        raise GPRError(f"libgpr_sm100a (multi-GPU) error {rc}: {msg.decode() if msg else ''}")

    def launch_count(self):
        return int(lib().gpr_mgpu_launch_count(self.handle))

    def set_option(self, name, value):
        self.check(lib().gpr_mgpu_set_option(self.handle, name.encode(), int(value)))

    def dbg_factor(self, A, Y=None, mode=0):
        A = np.array(A, dtype=np.float64, order="F")
        Yc = None if Y is None else np.array(Y, dtype=np.float64, order="F").reshape(A.shape[0], -1)
        info = _i64(0)
        ms = np.zeros(3)
        rc = lib().gpr_mgpu_dbg_factor(self.handle, dptr(A), A.shape[0], dptr(Yc), 0 if Yc is None else Yc.shape[1], int(mode),
                                       C.byref(info), dptr(ms))
        self.check(rc, info)
        return A, Yc, ms

    def close(self):
        if self._h is not None:
            lib().gpr_mgpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def dist_unique_id():
    """128-byte NCCL unique id (call on rank 0, ship the bytes to the other processes)."""
    buf = C.create_string_buffer(128)
    rc = lib().gpr_dist_unique_id(C.cast(buf, _vp))
    if rc != 0:
        msg = lib().gpr_mgpu_last_error(None)
        raise GPRError(f"gpr_dist_unique_id failed ({rc}): {msg.decode() if msg else ''}")
    return buf.raw


class DistContext(MultiContext):
    """One rank of a block-cyclic factorization that spans `world` PROCESSES (one GPU each, torchrun-style launch);
    panels travel over NCCL.  Same use as MultiContext afterwards (MultiModelHandle, nlml_grad on every rank)."""

    def __init__(self, device, rank, world, unique_id, nb=1024):
        self.devices, self.nb, self.rank, self.world = [int(device)], int(nb), int(rank), int(world)
        self._h = _vp()
        idbuf = C.create_string_buffer(bytes(unique_id), 128)
        rc = lib().gpr_dist_create(int(device), int(rank), int(world), C.cast(idbuf, _vp), self.nb, C.byref(self._h))
        if rc != 0:
            msg = lib().gpr_mgpu_last_error(None)
            self._h = None
            raise GPRError(f"gpr_dist_create(rank={rank}/{world}) failed ({rc}): {msg.decode() if msg else ''}")


class MultiModelHandle:
    """gpr_mgpu_model: x, y replicated, K / U / K^-1 block-cyclic over the ranks of a MultiContext."""

    def __init__(self, mctx, types, D, x, y, train_axis=1):
        self.mctx = mctx
        self.types = list(types)
        x = f64(x)
        y2 = f64(y.reshape(y.shape[0], -1))
        self.D, self.N = int(x.shape[0]), int(x.shape[1])
        self.ny = int(y2.shape[1])
        if D != self.D:
            raise GPRError("x dimension mismatch")
        if y2.shape[0] != self.N:
            raise GPRError("x and y size mismatch.")
        self.P = lib().gpr_dim_hp(types_array(self.types), len(self.types), self.D)
        self._h = _vp()
        rc = lib().gpr_mgpu_model_create(mctx.handle, types_array(self.types), len(self.types), self.D, self.N, dptr(x), dptr(y2),
                                         self.ny, int(train_axis), C.byref(self._h))
        if rc != 0:
            self._h = None
        mctx.check(rc)

    @property
    def handle(self):
        if self._h is None:
            raise GPRError("model destroyed")
        return self._h

    def nlml_grad(self, hp, log_scale=False, eps=1e-8, want_f=True, want_g=True):
        hp = f64(np.asarray(hp, dtype=np.float64).ravel())
        F = C.c_double(0.0)
        G = np.empty(self.P) if want_g else None
        info = _i64(0)
        rc = lib().gpr_mgpu_nlml_grad(self.handle, dptr(hp), hp.size, int(bool(log_scale)), float(eps),
                                      C.byref(F) if want_f else None, dptr(G), C.byref(info))
        self.mctx.check(rc, info)
        return (F.value if want_f else None), G

    def update_cache(self, hp, eps=1e-8, want_inverse=True):
        """gpr_mgpu_update_cache: the prediction needs K^-1, so want_inverse (the single-device signature) is always true here."""
        hp = f64(np.asarray(hp, dtype=np.float64).ravel())
        info = _i64(0)
        self.mctx.check(lib().gpr_mgpu_update_cache(self.handle, dptr(hp), hp.size, float(eps), C.byref(info)), info)

    def predict(self, xp, same_x=False, want_var=False, want_cov=False):
        xp = f64(xp)
        M = int(xp.shape[1])
        mean = np.empty((M, self.ny), order="F")
        var = np.empty(M) if want_var else None
        cov = np.empty((M, M), order="F") if want_cov else None
        self.mctx.check(lib().gpr_mgpu_predict(self.handle, dptr(xp), M, int(bool(same_x)), dptr(mean), dptr(var), dptr(cov)))
        return mean, var, cov

    def split_predict(self, xe, xq, var_range=None, want_var=True, mean_out=None, var_out=None):
        """gpr_mgpu_split_predict; arguments, results and in-place semantics as ModelHandle.split_predict"""
        xe, ne, xq, nq, lo, hi, mean, var = _split_args(xe, xq, var_range, want_var, mean_out, var_out)
        self.mctx.check(lib().gpr_mgpu_split_predict(self.handle, dptr(xe), ne, dptr(xq), nq, lo, hi, dptr(mean), dptr(var)))
        return mean, var

    def integrate(self, a, b, want_var=True):
        """gpr_mgpu_integrate.  a, b of shape (D,): (Iout (ny,), var (1,)) as ModelHandle.integrate; of shape (D, nbox):
        (Iout (nbox, ny), var (nbox,)), one pass over K^-1 for all boxes."""
        a, b, nbox, single = _box_args(a, b, self.D)
        Iout = np.empty((nbox, self.ny), order="F")
        var = np.empty(nbox) if want_var else None
        self.mctx.check(lib().gpr_mgpu_integrate(self.handle, nbox, dptr(a), dptr(b), dptr(Iout), dptr(var)))
        return (Iout[0], var) if single else (Iout, var)

    def fetch(self, which):
        out = np.empty((self.N, self.N), order="F") if which == FETCH_KINV else np.empty(self.N)
        self.mctx.check(lib().gpr_mgpu_fetch(self.handle, which, dptr(out)))
        return out

    def timings(self):
        ms = np.zeros(T_COUNT)
        self.mctx.check(lib().gpr_mgpu_timings(self.handle, dptr(ms), T_COUNT))
        return {n: float(ms[i]) for i, n in enumerate(T_NAMES)}

    def close(self):
        if self._h is not None:
            lib().gpr_mgpu_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
