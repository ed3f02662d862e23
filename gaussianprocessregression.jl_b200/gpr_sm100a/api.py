"""Host-side mirror of the reference's model / covariance / cost / predict API for the hot path.

Same names, argument meaning and error behaviour as srinix007/GaussianProcessRegression.jl (paths below are
relative to /root/reference); Julia's `f!` is spelled `f_`.  Everything numeric is done by libgpr_sm100a.so
through the C ABI (`_ffi.py`); this module holds no arithmetic beyond argument marshalling, the log-space
transform of `train` and the hyper-parameter bookkeeping the reference also does on the host.

Conventions kept from Julia: `x` is (D, N), `y` is (N,) or (N, ny), `kernel(cov, hp, x, xp)` is (N, M);
hyper-parameter indices `i` (grad) and `train_axis` are 1-based; `x === xp` is Python's `xp is x`.

The Julia glue that a maintainer of the reference would add (cache types holding the same handles and
`ccall`ing the same entry points) is julia/GPRsm100a.jl, described in INTEGRATION.md.
"""
import numpy as np

from . import _ffi
from ._ffi import GPRError, PosDefException, get_context  # noqa: F401


# --------------------------------------------------------------------------- covariance.jl / compose_covar.jl
class AbstractKernel:
    type_id = 0

    def __add__(self, other):
        """Base.:+ on kernels -> ComposedKernel (src/compose_covar.jl:9-19)"""
        a = self.kernels if isinstance(self, ComposedKernel) else (self,)
        b = other.kernels if isinstance(other, ComposedKernel) else (other,)
        return ComposedKernel(tuple(a) + tuple(b))

    def __eq__(self, other):
        return type(self) is type(other) and getattr(self, "kernels", None) == getattr(other, "kernels", None)

    def __hash__(self):
        return hash(type(self).__name__)

    def __repr__(self):
        return type(self).__name__ + "()"


class SquaredExp(AbstractKernel):
    """K(x,x') = sigma^2 exp(-|l .* (x - x')|^2), hp = [sigma, l_1..l_D]  (src/covariance.jl:4-15,85-95)"""
    type_id = _ffi.KERN_SE


class WhiteNoise(AbstractKernel):
    """sigma_n^2 * I on the self covariance only  (src/covariance.jl:17,60-64)"""
    type_id = _ffi.KERN_NOISE


class Matern52(AbstractKernel):
    """Extension, not in the reference (parity unpinned): sigma^2 (1 + sqrt5 r + 5 r^2/3) exp(-sqrt5 r), r = |l .* (x-x')|."""
    type_id = _ffi.KERN_MATERN52


class Euclidean:
    """src/covariance.jl:19"""


class ComposedKernel(AbstractKernel):
    """src/compose_covar.jl:1-3"""

    def __init__(self, kernels):
        self.kernels = tuple(kernels)

    def __repr__(self):
        return "(" + ", ".join(repr(k) for k in self.kernels) + ")"


def _components(cov):
    return list(cov.kernels) if isinstance(cov, ComposedKernel) else [cov]


def _types(cov):
    return [k.type_id for k in _components(cov)]


def dim_hp(cov, dim):
    """src/covariance.jl:27,60 ; src/compose_covar.jl:26-28"""
    return sum(1 if isinstance(k, WhiteNoise) else dim + 1 for k in _components(cov))


def split(hp, dims):
    """Base.split(A, inds)  (src/compose_covar.jl:21-24)"""
    c = np.concatenate([[0], np.cumsum(dims)])
    return [np.asarray(hp[c[i]:c[i + 1]]) for i in range(len(dims))]


def find_idx(dims, i):
    """src/compose_covar.jl:109-115 (1-based)"""
    cd = np.cumsum(dims)
    hit = np.nonzero(cd >= i)[0]
    kidx = int(hit[0]) + 1 if len(hit) else 0
    hpidx = i if kidx == 1 else i - int(cd[kidx - 2])
    return kidx, hpidx


class UniformScaling:
    """lambda * I (what grad(::WhiteNoise...) returns, src/deriv_covar.jl:31)"""

    def __init__(self, lam):
        self.λ = self.lam = float(lam)

    def __repr__(self):
        return f"UniformScaling({self.lam})"


def kernel(cov, hp, x, xp=None, dist=None, ϵ=1e-8, ctx=None):
    """kernel(K, hp, x[, xp]; ϵ)  (src/covariance.jl:29-47, src/compose_covar.jl:35-45).
    kernel(cov, hp, xp::Cmap, x) returns a `SplitKernel` (src/split_kernel.jl:125-135)."""
    if isinstance(x, Cmap):
        return _split_kernel(cov, hp, x, xp, ctx)
    x = np.asarray(x)
    if isinstance(cov, WhiteNoise):
        if xp is None:
            return UniformScaling(float(hp[0]) ** 2)       # hp[1]^2 * I  (src/covariance.jl:61)
        return 0.0
    ctx = ctx or get_context()
    if len(hp) != dim_hp(cov, x.shape[0]):
        raise GPRError("Parameter size mismatch.")
    if xp is None:
        # self form: jitter per component, noise on the diagonal for composed kernels
        return _ffi.kernel_matrix(ctx, _types(cov), x.shape[0], hp, x, x, True, ϵ, isinstance(cov, ComposedKernel))
    same = xp is x
    return _ffi.kernel_matrix(ctx, _types(cov), x.shape[0], hp, x, xp, same, ϵ, False)


def kernel_(kern, cov, hp, x, xp=None, ϵ=1e-8, ctx=None):
    """kernel!(kern, K, hp, x[, xp])  (src/covariance.jl:33-58, src/compose_covar.jl:47-77)"""
    if isinstance(kern, SplitKernel):
        new = _split_kernel(cov, hp, x, xp, ctx)      # kernel!(Kxps, cov, hp, xp::Cmap, x): x is the Cmap here
        kern.A[...], kern.B[...], kern.C[...] = new.A, new.B, new.C
        return None
    if isinstance(cov, WhiteNoise):
        return None
    kern[...] = kernel(cov, hp, x, xp, ϵ=ϵ, ctx=ctx)
    return None


def alloc_kernels(cov, x):
    """src/compose_covar.jl:90-100"""
    n = x.shape[1]
    return [np.zeros((1, 1)) if isinstance(k, WhiteNoise) else np.empty((n, n), order="F") for k in _components(cov)]


def kernels(cov, hp, x, ctx=None):
    """kernels(K, hp, x): list of per-component self covariances (src/compose_covar.jl:80-107)"""
    if not isinstance(cov, ComposedKernel):
        return [kernel(cov, hp, x, ctx=ctx)]
    dim = x.shape[0]
    hps = split(hp, [dim_hp(k, dim) for k in cov.kernels])
    return [np.zeros((1, 1)) if isinstance(k, WhiteNoise) else kernel(k, h, x, ctx=ctx) for k, h in zip(cov.kernels, hps)]


def add_noise_(kern, cov, hp, x):
    """src/compose_covar.jl:63-71 (host: N additions on the diagonal)"""
    comps = _components(cov)
    for idx, k in enumerate(comps):
        if isinstance(k, WhiteNoise):
            hps = split(hp, [dim_hp(c, x.shape[0]) for c in comps])
            kern[np.diag_indices(kern.shape[0])] += hps[idx][0] ** 2
            break
    return None


def rm_noise(cov, hps):
    """src/compose_covar.jl:30-33"""
    comps = _components(cov)
    return ([k for k in comps if not isinstance(k, WhiteNoise)],
            [h for k, h in zip(comps, hps) if not isinstance(k, WhiteNoise)])


def grad(cov_or_cost, *args, **kw):
    """grad(cov, i, hp, x) -> dK/dhp_i (src/deriv_covar.jl:2-18)   |   grad(cost, hp, md) (src/cost.jl:26-30)"""
    if isinstance(cov_or_cost, AbstractLoss):
        return _grad_cost(cov_or_cost, *args, **kw)
    return _grad_kernel(cov_or_cost, *args, **kw)


def _grad_kernel(cov, i, hp, x, K=None, ϵ=1e-8, ctx=None):
    dim = x.shape[0]
    if isinstance(cov, ComposedKernel):
        dims = [dim_hp(k, dim) for k in cov.kernels]
        hps = split(hp, dims)
        kidx, hpidx = find_idx(dims, i)
        return _grad_kernel(cov.kernels[kidx - 1], hpidx, hps[kidx - 1], x, ϵ=ϵ, ctx=ctx)
    if isinstance(cov, WhiteNoise):
        return UniformScaling(2.0 * float(hp[0]))           # src/deriv_covar.jl:31
    return _ffi.kernel_grad_matrix(ctx or get_context(), cov.type_id, dim, hp, x, i - 1, ϵ)


# --------------------------------------------------------------------------- models.jl
class GPRModel:
    """GPRModel(cov, hp, x, y; train_axis=1) / GPRModel(cov, x, y)  (src/models.jl:17-37)"""

    def __init__(self, cov, *args, train_axis=1):
        if len(args) == 3:
            hp, x, y = args
        elif len(args) == 2:
            x, y = args
            hp = np.random.rand(dim_hp(cov, np.asarray(x).shape[0]))
        else:
            raise TypeError("GPRModel(cov, [hp,] x, y)")
        x, y, hp = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64), np.asarray(hp, dtype=np.float64)
        if hp.shape[0] != dim_hp(cov, x.shape[0]):
            raise GPRError("Parameter size mismatch.")
        if x.shape[-1] != y.shape[0]:
            raise GPRError("x and y size mismatch.")
        self.covar, self.params, self.x, self.y, self.train_axis = cov, hp, x, y, int(train_axis)


def get_sample(md):
    """src/models.jl:39-45"""
    return md.y[:, md.train_axis - 1] if md.y.ndim == 2 else md.y


# --------------------------------------------------------------------------- loss_grad.jl / cost.jl / caches
class AbstractLoss:
    pass


class MarginalLikelihood(AbstractLoss):
    """src/loss_grad.jl:5"""


class LogScale:
    pass


class NoLogScale:
    pass


def islog(cost, md):
    """src/cost.jl:4-8"""
    if isinstance(cost, MarginalLikelihood):
        return LogScale() if any(isinstance(k, (SquaredExp, Matern52)) for k in _components(md.covar)) else NoLogScale()
    return NoLogScale()


class _DeviceCache:
    """Common part of the SM100 caches: one device-resident gpr_model per cache, like the reference's
    pre-allocated workspaces (src/caches/cost.jl, src/caches/predict.jl)."""
    want_inverse = False

    def __init__(self, md, ctx=None):
        self.ctx = ctx or get_context()
        self.hp = np.array(md.params, dtype=np.float64)
        self._x_ref, self._y_snapshot = md.x, np.array(md.y, copy=True)
        self.handle = _ffi.ModelHandle(self.ctx, _types(md.covar), md.x.shape[0], md.x, md.y, md.train_axis)

    def _sync_data(self, md):
        if md.x is not self._x_ref:
            self.handle.set_x(md.x)
            self._x_ref = md.x
        if not np.array_equal(md.y, self._y_snapshot):     # md.y .+= dy between calls (src/update_model.jl:36)
            self.handle.set_y(md.y)
            self._y_snapshot = np.array(md.y, copy=True)

    # cache internals pinned by test/test_loss.jl:46-48
    @property
    def kchol_base(self):
        return self.handle.fetch(_ffi.FETCH_U)

    @property
    def α(self):
        return self.handle.fetch(_ffi.FETCH_ALPHA)

    alpha = α

    @property
    def K_inv(self):
        return self.handle.fetch(_ffi.FETCH_KINV)

    @property
    def wt(self):
        w = self.handle.fetch(_ffi.FETCH_WT)
        return w[:, 0] if w.shape[1] == 1 else w

    def timings(self):
        return self.handle.timings()

    def close(self):
        self.handle.close()


class MllLossCache(_DeviceCache):
    """src/caches/cost.jl:6-19: hp, kchol_base, alpha"""
    want_inverse = False


class MllGradCache(_DeviceCache):
    """src/caches/cost.jl:21-44: additionally K^-1 (the per-component kernel list and dK buffer of the
    reference are never materialised here; the gradient kernel recomputes them on the fly)."""
    want_inverse = True


class MultiGPUGradCache:
    """Gradient cache whose K / U / K^-1 are block-cyclic over several ranks (one per entry of `devices`;
    default: every visible GPU once): BASELINE.json config 5, SURVEY.md 8e.  Drop-in for MllGradCache in
    loss_grad! / log_loss_grad! (src/cost.jl:50-70) and therefore in `train`.  After an evaluation with a gradient it
    also predicts (predict_mean_ / predict_, general test points or Cmap grids) at that evaluation's hyper-parameters;
    var_range: the rows e of a Cmap grid that get the posterior variance (1-based inclusive, as GPRSplitPredictCache)."""
    want_inverse = True

    def __init__(self, md, devices=None, nb=None, var_range=(1, 3)):
        self.var_range = var_range
        if devices is None:
            devices = list(range(max(1, _ffi.device_count())))
        if nb is None:
            # block-column width: 2048 once the matrix is large (the rank-nb products of potrf / trtri then run well on the INT8
            # tensor cores: N = 131072 on 8 B200 7.84 s against 8.69 s with 1024), 1024 below that (finer load balance)
            nb = 2048 if md.x.shape[1] >= 65536 else 1024
        self.mctx = _ffi.MultiContext(devices, nb=nb)
        self.hp = np.array(md.params, dtype=np.float64)
        self._x_ref, self._y_snapshot = md.x, np.array(md.y, copy=True)
        self.handle = _ffi.MultiModelHandle(self.mctx, _types(md.covar), md.x.shape[0], md.x, md.y, md.train_axis)

    def _sync_data(self, md):
        if md.x is not self._x_ref or not np.array_equal(md.y, self._y_snapshot):
            raise GPRError("MultiGPUGradCache: x / y changed; build a new cache")

    @property
    def α(self):
        return self.handle.fetch(_ffi.FETCH_ALPHA)

    alpha = α

    @property
    def K_inv(self):
        return self.handle.fetch(_ffi.FETCH_KINV)

    def timings(self):
        return self.handle.timings()

    def close(self):
        self.handle.close()
        self.mctx.close()


class MultiGPUPredictCache(MultiGPUGradCache):
    """Predict cache on the block-cyclic multi-GPU model (src/caches/predict.jl:3-31): update_cache_(pc, md) forms K^-1
    over the ranks (no gradient), predict_mean_ / predict_ (Diagonal and dense; Cmap grids with Diagonal) evaluate the
    posterior from it."""


def loss_cache(cost):
    return MllLossCache


def grad_cache(cost):
    return MllGradCache


def loss_grad_cache(cost):
    return MllGradCache


class GPRPredictCache(_DeviceCache):
    """src/caches/predict.jl:3-31 (Kxx, wt, Kxp live on the device)"""

    def __init__(self, md, xp=None, ctx=None):
        super().__init__(md, ctx)


class GPRSplitPredictCache(_DeviceCache):
    """src/caches/split_kernel.jl:1-30; var_range default 1:3 (1-based inclusive)"""

    def __init__(self, md, xp=None, var_range=(1, 3), ctx=None):
        super().__init__(md, ctx)
        self.var_range = var_range


def predict_cache(md, xp):
    """src/predict.jl:1, src/split_predict.jl:1"""
    return GPRSplitPredictCache if isinstance(xp, Cmap) else GPRPredictCache


def update_cache_(tc, *args, ϵ=1e-8):
    """update_cache!(tc, hp, md) (src/cost.jl:74-111)  |  update_cache!(pc, md) (src/predict.jl:29-34)"""
    if len(args) == 2:
        hp, md = args
    else:
        (md,) = args
        hp = md.params
    tc._sync_data(md)
    tc.hp = np.array(hp, dtype=np.float64)
    tc.handle.update_cache(tc.hp, eps=ϵ, want_inverse=tc.want_inverse)
    return None


def loss(cost, *args):
    """loss(cost, md) | loss(cost, hp, md) | loss(cost, hp, md, tc) | loss(cost, md, tc) | loss(cost, cov, hp, x, y)
    (src/cost.jl:17-22,40-43,113-117 ; src/loss_grad.jl:32-41)"""
    if not isinstance(cost, MarginalLikelihood):
        raise GPRError("only MarginalLikelihood is on the accelerated path")
    if len(args) == 1:
        md = args[0]
        return loss(cost, md.params, md)
    if len(args) == 2 and isinstance(args[1], _DeviceCache):
        md, tc = args
        return tc.handle.loss()
    if len(args) == 2:
        hp, md = args
        tc = loss_cache(cost)(md)
        try:
            return loss(cost, hp, md, tc)
        finally:
            tc.close()
    if len(args) == 3:
        hp, md, tc = args
        update_cache_(tc, hp, md)
        return tc.handle.loss()
    if len(args) == 4:                       # one-shot functional form: kernel -> cholesky -> \ -> formula
        cov, hp, x, y = args
        md = GPRModel(cov, hp, x, y)
        return loss(cost, hp, md)
    raise TypeError("loss: bad arguments")


def _grad_cost(cost, *args):
    if len(args) == 1:
        md = args[0]
        return _grad_cost(cost, md.params, md)
    hp, md = args
    G = np.empty(len(hp))
    grad_(G, cost, hp, md)
    return G


def grad_(dL, cost, *args):
    """grad!(dL, cost, hp, md) | grad!(dL, cost, hp, md, tc) | grad!(dL, cost, md, tc)  (src/cost.jl:32-48,119-127)"""
    if len(args) == 2 and isinstance(args[1], _DeviceCache):
        md, tc = args
        dL[...] = tc.handle.grad(False)
        return None
    if len(args) == 2:
        hp, md = args
        tc = grad_cache(cost)(md)
        try:
            grad_(dL, cost, hp, md, tc)
        finally:
            tc.close()
        return None
    hp, md, tc = args
    update_cache_(tc, hp, md)
    dL[...] = tc.handle.grad(False)
    return None


def loss_grad_(cost, F, G, hp, md, tc):
    """loss_grad!(cost, F, G, hp, md, tc): Optim only_fg! contract (src/cost.jl:50-58).
    F/G `None` means "not requested"; returns the loss iff F is not None; G is filled in place."""
    tc._sync_data(md)
    tc.hp = np.array(hp, dtype=np.float64)
    f, g = tc.handle.nlml_grad(tc.hp, log_scale=False, want_f=F is not None, want_g=G is not None)
    if G is not None:
        G[...] = g
    return f if F is not None else None


def log_loss_grad_(cost, F, G, log_hp, md, tc):
    """log_loss_grad!(cost, F, G, log_hp, md, tc)  (src/cost.jl:60-70): hp = exp.(log_hp); G .*= hp"""
    tc._sync_data(md)
    tc.hp = np.exp(np.asarray(log_hp, dtype=np.float64))
    f, g = tc.handle.nlml_grad(np.asarray(log_hp, dtype=np.float64), log_scale=True, want_f=F is not None,
                               want_g=G is not None)
    if G is not None:
        G[...] = g
    return f if F is not None else None


# --------------------------------------------------------------------------- train.jl
def init_params(cost, md):
    """src/train.jl:1-7"""
    if isinstance(cost, MarginalLikelihood):
        return np.ones_like(md.params)
    return np.random.rand(*md.params.shape)


def train(md, cost, hp0=None, method="L-BFGS-B", options=None):
    """train(md, cost, hp0; method, options)  (src/train.jl:9-87).

    The optimiser itself is the caller of the hot path and stays on the host (Optim.jl in the reference;
    scipy.optimize here because Julia is absent in this image).  What is mirrored exactly is the contract
    around it: log-space iff a SquaredExp is in the model (`islog`), `hp0` is then the LOG start point
    (default ones), one cache for the whole run, `fg!` = `log_loss_grad!`, result = exp.(minimizer)."""
    import scipy.optimize as so

    hp0 = init_params(cost, md) if hp0 is None else np.asarray(hp0, dtype=np.float64)
    log = isinstance(islog(cost, md), LogScale)
    tc = loss_grad_cache(cost)(md)
    fg = log_loss_grad_ if log else loss_grad_

    def fun(v):
        G = np.empty_like(v)
        f = fg(cost, True, G, v, md, tc)
        return f, G

    try:
        res = so.minimize(fun, hp0, jac=True, method=method, options=options or {})
    finally:
        tc.close()
    return (np.exp(res.x) if log else res.x), res


# --------------------------------------------------------------------------- predict.jl
class Diagonal:
    """LinearAlgebra.Diagonal stand-in: `.diag` vector."""

    def __init__(self, diag):
        self.diag = diag


def predict_mean(md, xp, ctx=None):
    """src/predict.jl:6-12"""
    pc = predict_cache(md, xp)(md, xp, ctx=ctx)
    try:
        update_cache_(pc, md)
        mu = np.empty(_mean_shape(md, xp), order="F")
        predict_mean_(mu, md, xp, pc)
        return mu
    finally:
        pc.close()


def _mean_shape(md, xp):
    if isinstance(xp, Cmap):
        return (xp.xe.shape[1], xp.xq.shape[1])
    M = xp.shape[1]
    return (M,) if md.y.ndim == 1 else (M, md.y.shape[1])


def predict(md, xp, diagonal_var=False, ctx=None):
    """src/predict.jl:14-25: returns (mu, Sigma) with Sigma dense (M, M) or Diagonal"""
    pc = predict_cache(md, xp)(md, xp, ctx=ctx)
    try:
        update_cache_(pc, md)
        mu = np.empty(_mean_shape(md, xp), order="F")
        nflat = int(np.prod(mu.shape))
        if not diagonal_var:
            if isinstance(xp, Cmap):
                raise GPRError("split predict supports diagonal_var=true only (src/split_predict.jl:39)")
            Sig = np.empty((xp.shape[1], xp.shape[1]), order="F")
        else:
            Sig = Diagonal(np.empty(nflat))
        predict_(mu, Sig, md, xp, pc)
        return mu, Sig
    finally:
        pc.close()


def _inplace(a, shape, order):
    """`a` itself if the C ABI can write the result straight into it (float64, right shape, dense in the given order)."""
    ok = isinstance(a, np.ndarray) and a.dtype == np.float64 and a.shape == tuple(shape) and a.flags.writeable and \
        (a.flags.f_contiguous if order == "F" else a.flags.c_contiguous)
    return a if ok else None


def predict_mean_(mu, md, xp, pc):
    """predict_mean!(mu, md, xp, pc)  (src/predict.jl:36-40 ; split: src/split_predict.jl:5-19)"""
    if isinstance(xp, Cmap):
        out = _inplace(mu, (xp.xe.shape[1], xp.xq.shape[1]), "F")          # written in place when the layout allows it
        m, _ = pc.handle.split_predict(xp.xe, xp.xq, var_range=None, want_var=False, mean_out=out)
        if out is None:
            mu[...] = m
        return None
    m, _, _ = pc.handle.predict(xp, same_x=xp is md.x)
    mu[...] = m.reshape(mu.shape, order="F")
    return None


def predict_(mu, Sig, md, xp, pc):
    """predict!(mu, Sigma, md, xp, pc) -- dense, Diagonal and Cmap methods (src/predict.jl:42-71)"""
    if isinstance(xp, Cmap):
        if not isinstance(Sig, Diagonal):
            raise GPRError("split predict supports Diagonal covariance only")
        ne, nq = xp.xe.shape[1], xp.xq.shape[1]
        out, vout = _inplace(mu, (ne, nq), "F"), _inplace(Sig.diag, (ne * nq,), "C")
        m, v = pc.handle.split_predict(xp.xe, xp.xq, var_range=pc.var_range, want_var=True, mean_out=out, var_out=vout)
        if out is None:
            mu[...] = m
        if vout is None:
            Sig.diag[...] = v
        return None
    same = xp is md.x
    if isinstance(Sig, Diagonal):
        m, v, _ = pc.handle.predict(xp, same_x=same, want_var=True)
        Sig.diag[...] = v
    else:
        m, _, c = pc.handle.predict(xp, same_x=same, want_var=True, want_cov=True)
        Sig[...] = c
    mu[...] = m.reshape(mu.shape, order="F")
    return None


# --------------------------------------------------------------------------- split_kernel.jl
class Cmap:
    """Cmap(op, xe, xq): lazy op.(xe[:, e], xq[:, q]), size (D, ne, nq)  (src/split_kernel.jl:1-17).
    The split factorisation is valid for op = + only (src/split_kernel.jl:151-159)."""

    def __init__(self, op, xe, xq):
        self.op, self.xe, self.xq = op, np.asarray(xe, dtype=np.float64), np.asarray(xq, dtype=np.float64)

    @property
    def shape(self):
        return (self.xe.shape[0], self.xe.shape[1], self.xq.shape[1])

    def __getitem__(self, idx):
        """xeq[i, j] (0-based ints or slices); xeq[:, :] flattens with e fastest (test/test_split_kernel.jl:20-21)."""
        i, j = idx
        xe = self.xe[:, i] if not isinstance(i, slice) else self.xe[:, i]
        xq = self.xq[:, j] if not isinstance(j, slice) else self.xq[:, j]
        xe = xe.reshape(self.xe.shape[0], -1)
        xq = xq.reshape(self.xq.shape[0], -1)
        out = self.op(xe[:, :, None], xq[:, None, :])
        return out.reshape(self.xe.shape[0], -1, order="F")


class SplitKernel:
    """A (ne, nq, k), B (ne, N, k), C (N, nq, k); K[e, q, s] = sum_k A B C  (src/split_kernel.jl:19-105)"""

    def __init__(self, A, B, C):
        self.A, self.B, self.C = A, B, C

    @property
    def shape(self):
        return (self.A.shape[0], self.A.shape[1], self.C.shape[0], self.A.shape[2])

    def __getitem__(self, idx):
        e, q, s = idx
        return np.einsum("...k,...k,...k->...", self.A[e, q, :], self.B[e, s, :], self.C[s, q, :])


def _split_kernel(cov, hp, xeq, x, ctx=None):
    ctx = ctx or get_context()
    if xeq.op is not np.add and getattr(xeq.op, "__name__", "") not in ("add", "<lambda>"):
        raise GPRError("SplitKernel is defined for Cmap(+, xe, xq) only")
    A, B, C = _ffi.split_kernel_arrays(ctx, _types(cov), x.shape[0], hp, xeq.xe, xeq.xq, x)
    return SplitKernel(A, B, C)


# =========================================================================== SURVEY.md 8f "next" rows: callers of the hot path
# Host logic exactly as in the reference (these drivers are Julia code there too); every factorization, solve,
# gradient and prediction they issue goes through the same device entry points as above.

# --------------------------------------------------------------------------- loss_grad.jl:6-30 (M-estimators)
class MSE(AbstractLoss):
    """src/loss_grad.jl:6,11-14"""


class ChiSq(AbstractLoss):
    """src/loss_grad.jl:7,16-22"""


class Mahalanobis(AbstractLoss):
    """src/loss_grad.jl:8,24-29"""


def m_loss(cost, y, yp, Σp):
    """loss(::MSE | ::ChiSq | ::Mahalanobis, y, yp, Σp)  (src/loss_grad.jl:11-29).  ntst-sized host arithmetic."""
    y, yp = np.asarray(y, dtype=np.float64), np.asarray(yp, dtype=np.float64)
    if isinstance(cost, MSE):
        return float(np.sum((y - yp) ** 2) / len(y))
    S = Σp.diag if isinstance(Σp, Diagonal) else np.asarray(Σp)
    if isinstance(cost, ChiSq):
        d = S if S.ndim == 1 else np.diag(S)
        return float(np.sum((y - yp) ** 2 / d))
    if isinstance(cost, Mahalanobis):
        import scipy.linalg as sl
        dl = sl.solve_triangular(sl.cholesky(S, lower=True), y - yp, lower=True)
        return float(dl @ dl)
    raise TypeError("m_loss: unknown cost")


# --------------------------------------------------------------------------- crossval.jl
def kfoldcv(n, k, nb=None, rng=None):
    """kfoldcv(n, k, nb = div(n, k))  (src/crossval.jl:1-12); 0-based indices"""
    nb = n // k if nb is None else nb
    nsh = (rng or np.random.default_rng()).permutation(n)
    trn, tst = [], []
    for i in range(nb):
        idx = np.arange(i * k, (i + 1) * k)
        tst.append(nsh[idx])
        trn.append(np.delete(nsh, idx))
    return trn, tst


def cv_step_(cost, mdt, xtst, ytst, pc, yp, Σp):
    """cv_step!(cost, mdt, xtst, ytst, pc, yp, Σp)  (src/crossval.jl:45-50)"""
    update_cache_(pc, mdt)
    predict_(yp, Σp, mdt, xtst, pc)
    return m_loss(cost, ytst, yp, Σp)


def cv_step(md, cost, xtr, ytr, xtst, ytst):
    """cv_step(md, cost, xtr, ytr, xtst, ytst)  (src/crossval.jl:37-43)"""
    mdt = GPRModel(md.covar, md.params, xtr, ytr)
    pc = predict_cache(mdt, xtst)(mdt, xtst)
    yp = np.empty(np.asarray(ytst).shape[0])
    Σp = np.empty((yp.shape[0], yp.shape[0]), order="F")
    try:
        return cv_step_(cost, mdt, xtst, ytst, pc, yp, Σp)
    finally:
        pc.close()


def cv_batch(md, cost, x, y, cvset):
    """cv_batch(md, cost, x, y, cvset)  (src/crossval.jl:14-35): one device model re-used across the folds (every fold
    has the same training size, as in the reference, which overwrites mdt.x / mdt.y in place)."""
    trn, tst = cvset
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    ntst = len(tst[0])
    yp = np.empty(ntst)
    Σp = np.empty((ntst, ntst), order="F")
    lss = np.empty(len(trn))
    mdt = GPRModel(md.covar, md.params, np.asfortranarray(x[:, trn[0]]), y[trn[0]].copy())
    pc = predict_cache(mdt, x[:, tst[0]])(mdt, None)
    try:
        for i in range(len(trn)):
            mdt.x = np.asfortranarray(x[:, trn[i]])      # a new object: the cache re-uploads it (md.x is compared by identity)
            mdt.y = y[trn[i]].copy()
            lss[i] = cv_step_(cost, mdt, np.asfortranarray(x[:, tst[i]]), y[tst[i]], pc, yp, Σp)
    finally:
        pc.close()
    return lss


# --------------------------------------------------------------------------- update_model.jl
class BFGSQuad:
    """src/update_model.jl:2"""


class BFGSQuadCache:
    """src/caches/update_model.jl:4-20: hp (log space), J, hess_inv"""

    def __init__(self, md):
        n = len(md.params)
        self.hp, self.J, self.hess_inv = np.empty(n), np.empty(n), np.empty((n, n))


def updater_cache(upd):
    return BFGSQuadCache


def bfgs_hessian(Bi, s, t, ρ=None):
    """bfgs_hessian(Bi, s, t, ρ = 1 / dot(s, t))  (src/update_model.jl:50-54); Bi = None stands for `I`"""
    s, t = np.asarray(s, dtype=np.float64), np.asarray(t, dtype=np.float64)
    ρ = 1.0 / float(s @ t) if ρ is None else ρ
    n = len(s)
    Bi = np.eye(n) if Bi is None else np.asarray(Bi)
    Cm = np.eye(n) - ρ * np.outer(s, t)
    B = Cm @ Bi @ Cm.T + ρ * np.outer(s, s)
    return 0.5 * (B + B.T)


def bfgs_quad_(θ, JJ, B, gradL, ϵ, max_iter=100):
    """bfgs_quad!(θ, JJ, B, ∇L, ϵ, max_iter)  (src/update_model.jl:64-79)"""
    it = 0
    while np.linalg.norm(JJ) > ϵ and it < max_iter:
        s, t = θ.copy(), JJ.copy()
        θ -= B @ JJ
        JJ[...] = gradL(θ)
        s, t = θ - s, JJ - t
        B[...] = bfgs_hessian(B, s, t)
        it += 1
    return it


def bfgs_quad(xx, JJ, HH, jac, ϵ=1e-5, max_iter=100):
    """bfgs_quad(xx, JJ, HH, jac; ϵ, max_iter)  (src/update_model.jl:56-62); HH = None stands for `I`"""
    x0, J0 = np.array(xx, dtype=np.float64), np.array(JJ, dtype=np.float64)
    B = np.eye(len(x0)) if HH is None else np.linalg.inv(HH)
    it = bfgs_quad_(x0, J0, B, jac, ϵ, max_iter)
    return x0, J0, np.linalg.inv(B), it


def hessian_fd_(hess, gradL, x, ϵ=1e-6):
    """hessian_fd!(hess, ∇L, x, ϵ)  (src/update_model.jl:87-94): P + 1 independent gradient evaluations.  If ∇L has a
    `many(list_of_points) -> list_of_gradients` attribute (ReplicaGradient below: one evaluation per GPU at a time,
    SURVEY.md 8e "replicas"), the P + 1 points are evaluated through it in one batch."""
    x = np.asarray(x, dtype=np.float64)
    pts = [x.copy()]
    for i in range(len(x)):
        xe = x.copy()
        xe[i] += ϵ
        pts.append(xe)
    gs = gradL.many(pts) if hasattr(gradL, "many") else [gradL(p) for p in pts]
    for i in range(len(x)):
        hess[:, i] = (gs[i + 1] - gs[0]) / ϵ
    return hess


def hessian_fd(gradL, x, ϵ=1e-6):
    """hessian_fd(∇L, x, ϵ)  (src/update_model.jl:81-85)"""
    n = len(x)
    return hessian_fd_(np.empty((n, n)), gradL, x, ϵ)


class ReplicaGradient:
    """∇L closure of update_sample! (`jj`, src/update_model.jl:21-27,38-44) over one gradient cache per device:
    `many(points)` spreads independent hyper-parameter points over the devices (one host thread per device; the C
    calls release the GIL and distinct contexts may be used from distinct threads), a plain call uses device 0."""

    def __init__(self, cost, md, caches):
        self.cost, self.md, self.caches = cost, md, list(caches)

    def __call__(self, log_x):
        G = np.empty(len(log_x))
        log_loss_grad_(self.cost, None, G, log_x, self.md, self.caches[0])
        return G

    def many(self, points):
        from concurrent.futures import ThreadPoolExecutor
        n = len(self.caches)
        if n == 1:
            return [self(p) for p in points]
        out = [None] * len(points)

        def work(w):
            for i in range(w, len(points), n):
                G = np.empty(len(points[i]))
                log_loss_grad_(self.cost, None, G, points[i], self.md, self.caches[w])
                out[i] = G

        with ThreadPoolExecutor(n) as ex:
            list(ex.map(work, range(n)))
        return out


def update_cache_bfgs_(uc, md, cost, tc, replicas=None):
    """update_cache!(uc::BFGSQuadCache, md, cost, tc)  (src/update_model.jl:18-32)"""
    uc.hp[...] = np.log(md.params)
    jac = ReplicaGradient(cost, md, [tc] + list(replicas or []))
    uc.J[...] = jac(uc.hp)
    hess = hessian_fd(jac, uc.hp)
    uc.hess_inv[...] = np.linalg.inv(np.triu(hess) + np.triu(hess, 1).T)      # inv(Hermitian(hess)): upper triangle
    return jac


def update_sample_(md, δy, *args, replicas=None):
    """update_sample!(md, δy, upd, cost[, ϵJ]) | update_sample!(md, δy, cost, uc, tc[, ϵJ])  (src/update_model.jl:8-48):
    md.y .+= δy, then a quasi-Newton re-optimisation of the log hyper-parameters started from the gradient and the
    finite-difference Hessian at the current (previously optimal) point.  `replicas`: extra gradient caches on other
    devices for the P + 1 evaluations of the Hessian.  Returns the number of iterations."""
    if isinstance(args[0], BFGSQuad):
        cost = args[1]
        ϵJ = args[2] if len(args) > 2 else 1e-3
        md.y += δy
        tc = grad_cache(cost)(md)
        uc = updater_cache(args[0])(md)
        try:
            return _update_sample_core(md, cost, uc, tc, ϵJ, replicas)
        finally:
            tc.close()
    cost, uc, tc = args[0], args[1], args[2]
    ϵJ = args[3] if len(args) > 3 else 1e-3
    md.y += δy
    return _update_sample_core(md, cost, uc, tc, ϵJ, replicas)


def _update_sample_core(md, cost, uc, tc, ϵJ, replicas):
    for c in [tc] + list(replicas or []):
        c._sync_data(md)
    jac = update_cache_bfgs_(uc, md, cost, tc, replicas)
    iters = bfgs_quad_(uc.hp, uc.J, uc.hess_inv, jac, ϵJ)
    md.params[...] = np.exp(uc.hp)
    return iters


# --------------------------------------------------------------------------- distributions.jl
class NormalDistribution:
    """src/distributions.jl:4-9,20-28.  Holds what `sample` needs: the covariance spec instead of a dense Σ."""

    def __init__(self, μ, cov, θ, x):
        self.μ, self.cov, self.θ, self.x = μ, cov, np.asarray(θ, dtype=np.float64), np.asarray(x, dtype=np.float64)


class GaussianProcess:
    """GaussianProcess(f_μ, kernel); gp(x[, θ]) -> NormalDistribution  (src/distributions.jl:11-14,37-46)"""

    def __init__(self, f_μ, kernel):
        self.f_μ, self.kernel = f_μ, kernel

    def __call__(self, x, θ=None):
        x = np.asarray(x, dtype=np.float64)
        if θ is None:
            θ = np.random.rand(dim_hp(self.kernel, x.shape[0]))
        μ = np.array([self.f_μ(x[:, j]) for j in range(x.shape[1])], dtype=np.float64)
        return NormalDistribution(μ, self.kernel, θ, x)


def sample(dist_or_gp, *args, rng=None, z=None, ctx=None):
    """sample(N::NormalDistribution; rng) | sample(gp, x[, θ])  (src/distributions.jl:30-35):
    s = cholesky(Σ .+ 1e-7).L * randn(rng, dim) .+ μ with Σ = kernel(cov, θ, x).  The draws come from `rng`
    (numpy Generator; the reference uses Xoshiro(1)) or are passed explicitly as `z`; the factorization and the
    product run on the device (gpr_sample_mvn)."""
    N = dist_or_gp(*args) if isinstance(dist_or_gp, GaussianProcess) else dist_or_gp
    n = N.x.shape[1]
    if z is None:
        z = (rng or np.random.default_rng(1)).standard_normal(n)
    return _ffi.sample_mvn(ctx or get_context(), _types(N.cov), N.x.shape[0], N.θ, N.x, z, N.μ, 1e-7)


# --------------------------------------------------------------------------- integrate.jl (noise-free path)
_RT_PI_BY_2 = 0.5 * np.sqrt(np.pi)


def _erf2(x, y):
    """SpecialFunctions.erf(x, y) = erf(y) - erf(x) without cancellation"""
    import scipy.special as sp
    x, y = np.broadcast_arrays(np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64))
    r = 1.0 / np.sqrt(2.0)
    small = (np.abs(x) <= r) & (np.abs(y) <= r)
    out = sp.erf(y) - sp.erf(x)
    out = np.where((x >= 0) & (y >= 0) & ~small, sp.erfc(x) - sp.erfc(y), out)
    out = np.where((x <= 0) & (y <= 0) & ~small, sp.erfc(-y) - sp.erfc(-x), out)
    return out


def gauss_integ(xs, w, a, b):
    """gauss_integ(xs, w, a, b)  (src/integrate.jl:4-5)"""
    return (1.0 / w) * _RT_PI_BY_2 * _erf2(w * (a - xs), w * (b - xs))


def erf_integ(w, a, b):
    """erf_integ(w, a, b)  (src/integrate.jl:6-7)"""
    import scipy.special as sp
    return 1.0 / (w ** 2) * (np.exp(-(w * (b - a)) ** 2) - 1.0) + 2.0 * (_RT_PI_BY_2 / w) * (b - a) * sp.erf(w * (b - a))


def antideriv2(cov, hp, a, b):
    """antideriv2(::SquaredExp, hp, a, b)  (src/integrate.jl:33-41)"""
    dim = len(a)
    ls = np.asarray(hp[1:dim + 1], dtype=np.float64)
    return float(np.prod(erf_integ(ls, np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64))) * hp[0] ** 2)


def integrate(md, *args, sample_noise=None, ctx=None, cache=None):
    """integrate(md, a, b; sample_noise) | integrate(md, hp, a, b; sample_noise)  (src/integrate.jl:45-62):
    mean and variance of the integral of the posterior over the box [a, b].  Returns (Iout[ny], var_Iout).

    sample_noise = nothing: Cholesky path (:65-70,131-136), var_Iout has one entry.
    sample_noise = scalar / vector (one extra diagonal noise per column of y): the reference diagonalises K once (LAPACK
    syevr, :72-80) and applies (K + eps_i I)^-1 = P (lambda + eps_i)^-1 P' per column.  The device has no symmetric
    eigensolver; the SAME quantities -- mu_i = y_i' (K + eps_i I)^-1 k1 and var_i = k2 - k1' (K + eps_i I)^-1 k1 -- are
    obtained from one shifted Cholesky factorization per distinct noise level (the shift rides in the jitter argument of
    update_cache!), i.e. N^3/3 flop per level instead of one ~9 N^3 eigendecomposition: cheaper up to ~27 levels.

    a, b may also be D x nbox arrays (box i = column i): Iout is then (nbox, ny) and var_Iout (nbox,) -- (nbox, ny) with
    sample_noise, one row per box as the single-box call returns it.
    cache: a MultiGPUGradCache / MultiGPUPredictCache of md; the factorizations then run block-cyclic on its devices
    (update_cache_ on that cache) and all boxes go through gpr_mgpu_integrate in one pass over K^-1.  Without it, one
    device: gpr_integrate for a single box, and gpr_integrate_batch for all boxes of a D x nbox batch in one call per
    factorization (one triangular solve per tile of boxes)."""
    if len(args) == 2:
        hp, (a, b) = md.params, args
    else:
        hp, a, b = args
    multi = isinstance(cache, MultiGPUGradCache)
    a2, b2 = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    batched = a2.ndim == 2
    wc = cache if multi else MllLossCache(md, ctx)

    def once(eps):
        update_cache_(wc, hp, md, ϵ=eps)
        return wc.handle.integrate(a2, b2, want_var=True)

    try:
        if sample_noise is None:
            return once(1e-8)
        ny = 1 if md.y.ndim == 1 else md.y.shape[1]
        # the jitter is added once per non-noise component (src/compose_covar.jl:53-55), so eps_i is split among them
        nk = sum(1 for k in _components(md.covar) if not isinstance(k, WhiteNoise))
        if np.ndim(sample_noise) == 0:
            Iout, var = once(1e-8 + float(sample_noise) / nk)
            return Iout, np.repeat(var[:, None], ny, axis=1) if batched else np.full(ny, var[0])   # var_Iout .= k2 .- scalar  (:157-158)
        noise = np.asarray(sample_noise, dtype=np.float64).ravel()
        if noise.size != ny:
            raise GPRError("sample_noise needs one entry per column of y")
        nbox = a2.shape[1] if batched else 1
        Iout, var = np.empty((nbox, ny)), np.empty((nbox, ny))
        done = {}
        for i, e in enumerate(noise):
            if e not in done:
                done[e] = once(1e-8 + float(e) / nk)
            Ii, vi = done[e]
            Iout[:, i], var[:, i] = Ii.reshape(nbox, ny)[:, i], vi
        return (Iout, var) if batched else (Iout[0], var[0])
    finally:
        if not multi:
            wc.close()
