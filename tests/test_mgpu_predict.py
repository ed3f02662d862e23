"""Posterior prediction on the block-cyclic multi-GPU model (gpr_mgpu_update_cache / gpr_mgpu_predict, pytest -m gpu).
The ranks cycle over the visible GPUs, so a 1-GPU box runs the whole distributed path with several ranks on cuda:0.

Tolerances as in tests/test_gpu_parity.py: mean rel 1e-8 against max(|mu|, 1e-8 |y|_inf), variance and covariance abs
1e-8 * sum sigma^2, either raised to 10 cond(K) eps where that is larger."""
import ctypes
import os

import numpy as np
import pytest

import gpr_oracle as o

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
EPS = 2.2e-16
TOL_MU, TOL_VAR = 1e-8, 1e-8


def _devices(G):
    from gpr_sm100a import _ffi
    nd = max(1, _ffi.device_count())
    return [r % nd for r in range(G)]


def to_gpr_cov(gpr, cov):
    m = {o.SE: gpr.SquaredExp, o.NOISE: gpr.WhiteNoise, o.MATERN52: gpr.Matern52}
    k = m[cov[0]]()
    for c in cov[1:]:
        k = k + m[c]()
    return k


def ctol(stated, cond):
    return max(stated, 10.0 * cond * EPS)


def mean_err(mu, ref, y):
    return float((np.abs(mu - ref) / np.maximum(np.abs(ref), 1e-8 * np.abs(y).max())).max())


def problem(cov, N, D, ny, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    if ny > 1:
        y = np.stack([y * (0.5 + 0.3 * k) for k in range(ny)], axis=1)
    hp = 0.3 + rng.random(o.dim_hp(cov, D))
    hp[-1] = 0.1
    return x, y, hp, rng


def predict_all(pc, md, xp, dense=True):
    """predict_mean_, predict_ (Diagonal) and, optionally, predict_ (dense) through the mirrored host API"""
    import gpr_sm100a as gpr
    M = xp.shape[1]
    shape = (M,) if md.y.ndim == 1 else (M, md.y.shape[1])
    mu0 = np.empty(shape, order="F")
    gpr.predict_mean_(mu0, md, xp, pc)
    mu = np.empty(shape, order="F")
    Sd = gpr.Diagonal(np.empty(M))
    gpr.predict_(mu, Sd, md, xp, pc)
    assert np.array_equal(mu0, mu)
    if not dense:
        return mu, Sd.diag, None
    mu2 = np.empty(shape, order="F")
    Sf = np.empty((M, M), order="F")
    gpr.predict_(mu2, Sf, md, xp, pc)
    assert np.array_equal(mu2, mu)
    return mu, Sd.diag, Sf


def check_oracle(mdo, xp, mu, var, Sf, y, cond, same=False):
    prior = o.prior_diag(mdo)
    mu_o, var_o = o.predict(mdo, xp, diagonal_var=True, same=same)
    assert mean_err(mu.reshape(mu_o.shape), mu_o, y) <= ctol(TOL_MU, cond)
    assert np.abs(var - var_o).max() <= ctol(TOL_VAR, cond) * prior
    if Sf is not None:
        _, S_o = o.predict(mdo, xp, same=same)
        assert np.abs(Sf - S_o).max() <= ctol(TOL_VAR, cond) * prior


# (composition, N, D, ny, nb, G): N = 300 with nb = 128 on 8 ranks leaves ranks without a block; N is no multiple of nb
CASES = [((o.SE, o.NOISE), 300, 3, 1, 128, 8), ((o.SE, o.NOISE), 1000, 5, 3, 256, 2), ((o.SE, o.SE, o.NOISE), 1000, 4, 1, 128, 3),
         ((o.SE, o.MATERN52, o.NOISE), 2000, 6, 1, 256, 3), ((o.SE, o.NOISE), 2000, 8, 1, 128, 1),
         ((o.SE, o.SE, o.NOISE), 300, 2, 3, 256, 2), ((o.SE, o.MATERN52, o.NOISE), 1000, 3, 1, 128, 8)]


@pytest.mark.parametrize("cov,N,D,ny,nb,G", CASES)
def test_mgpu_predict_vs_oracle(gpr, cov, N, D, ny, nb, G):
    x, y, hp, rng = problem(cov, N, D, ny, N + 7 * G + nb)
    ta = 2 if ny > 1 else 1
    mdo = o.GPRModel(cov, hp, x, y, train_axis=ta)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    md = gpr.GPRModel(to_gpr_cov(gpr, cov), hp, x, y, train_axis=ta)
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(G), nb=nb)
    gpr.update_cache_(pc, md)
    for M in (1, 127, 1000):
        xp = rng.random((D, M))
        mu, var, Sf = predict_all(pc, md, xp)
        check_oracle(mdo, xp, mu, var, Sf, y, cond)
    # tiles: predict_tile forced to 128, M = 300 -> three tiles
    pc.mctx.set_option("predict_tile", 128)
    xp = rng.random((D, 300))
    mu, var, _ = predict_all(pc, md, xp, dense=False)
    check_oracle(mdo, xp, mu, var, None, y, cond)
    # xp === md.x: the training points themselves (jitter on the diagonal of K(x, xp))
    mu, var, Sf = predict_all(pc, md, md.x)
    check_oracle(mdo, x, mu, var, Sf, y, cond, same=True)
    pc.close()


def _cond_bound(K, floor):
    """cond_2(K) <= lambda_max / (sigma_n^2 + jitter): the smallest eigenvalue is at least the noise floor"""
    import scipy.sparse.linalg as sla
    return float(sla.eigsh(K, k=1, which="LA", return_eigenvectors=False)[0]) / floor


@pytest.mark.parametrize("ozaki", [0, -1])
def test_mgpu_predict_matches_single_gpu_n8192(gpr, ozaki):
    """Config 2 set A (N = 8192, D = 8, SE + noise): the explicit-inverse quadratic form on 4 ranks against the single-GPU
    triangular solve, DMMA products (ozaki 0) and the automatic route."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mg2", os.path.join(HERE, "golden", "make_golden_config2.py"))
    mg2 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg2)
    x, y, sets = mg2.inputs()
    hp = sets["A"]
    rng = np.random.default_rng(82)
    xp = rng.random((x.shape[0], 2048))
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    ref = gpr.GPRPredictCache(md)
    gpr.update_cache_(ref, md)
    mu_r, var_r, _ = ref.handle.predict(xp, want_var=True)
    _, _, S_r = ref.handle.predict(xp[:, :512], want_cov=True)
    ref.close()
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(4), nb=512)
    pc.mctx.set_option("ozaki", ozaki)
    gpr.update_cache_(pc, md)
    mu, var, _ = pc.handle.predict(xp, want_var=True)
    _, _, S = pc.handle.predict(xp[:, :512], want_cov=True)
    pc.close()
    cond = _cond_bound(o.kernel((o.SE, o.NOISE), hp, x), hp[-1] ** 2 + 1e-8)
    prior = hp[0] ** 2 + hp[-1] ** 2
    em, ev, es = mean_err(mu, mu_r, y), np.abs(var - var_r).max() / prior, np.abs(S - S_r).max() / prior
    print(f"\nN = 8192 on 4 ranks, ozaki {ozaki}: cond <= {cond:.1e}, mean {em:.1e}, var {ev:.1e}, cov {es:.1e}")
    assert em <= ctol(TOL_MU, cond) and ev <= ctol(TOL_VAR, cond) and es <= ctol(TOL_VAR, cond)


def test_mgpu_predict_deterministic_and_transports(gpr):
    """Transport 0 (peer reads) and transport 1 (pack -> collective -> unpack) give bit-identical outputs; two calls give
    identical outputs; the prediction leaves K^-1 untouched."""
    from gpr_sm100a import _ffi
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 1000, 4, 1, 5)
    xp = rng.random((4, 700))
    outs = []
    for transport in (0, 1):
        mc = _ffi.MultiContext(_devices(3), nb=128, transport=transport)
        mm = _ffi.MultiModelHandle(mc, [1, 2], 4, x, y)
        mm.update_cache(hp)
        K0 = mm.fetch(_ffi.FETCH_KINV)
        a = mm.predict(xp, want_var=True, want_cov=True)
        b = mm.predict(xp, want_var=True, want_cov=True)
        assert all(np.array_equal(u, v) for u, v in zip(a, b))
        assert np.array_equal(mm.fetch(_ffi.FETCH_KINV), K0)
        t = mm.timings()
        assert t["pred_kstar"] > 0 and t["pred_trsm"] > 0 and t["pred_rownorm"] > 0 and t["pred_mean"] > 0, t
        outs.append(a)
        mm.close(); mc.close()
    assert all(np.array_equal(u, v) for u, v in zip(outs[0], outs[1]))


def test_mgpu_predict_ready_by_update_cache_or_gradient(gpr):
    """gpr_mgpu_update_cache and gpr_mgpu_nlml_grad with G leave the same K^-1: the same outputs at the same hp."""
    import gpr_sm100a as g
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 900, 3, 1, 11)
    xp = rng.random((3, 400))
    md = g.GPRModel(to_gpr_cov(gpr, cov), hp, x, y)
    pc = g.MultiGPUPredictCache(md, devices=_devices(2), nb=128)
    g.update_cache_(pc, md)
    a = pc.handle.predict(xp, want_var=True, want_cov=True)
    pc.close()
    tc = g.MultiGPUGradCache(md, devices=_devices(2), nb=128)
    G = np.empty(len(hp))
    g.loss_grad_(g.MarginalLikelihood(), True, G, hp, md, tc)
    b = tc.handle.predict(xp, want_var=True, want_cov=True)
    tc.close()
    assert all(np.array_equal(u, v) for u, v in zip(a, b))


def test_mgpu_predict_errors(gpr):
    from gpr_sm100a import _ffi
    x, y, hp, rng = problem((o.SE, o.NOISE), 500, 2, 1, 3)
    xp = rng.random((2, 10))
    mc = _ffi.MultiContext(_devices(2), nb=128)
    mm = _ffi.MultiModelHandle(mc, [1, 2], 2, x, y)
    L = _ffi.lib()
    GPR_ERR_ARG, GPR_ERR_STATE = -1, -4

    def rc_predict(xp_, M, same=0):
        mean = np.empty(max(M, 1))
        return L.gpr_mgpu_predict(mm.handle, None if xp_ is None else _ffi.dptr(xp_), M, same, _ffi.dptr(mean), None, None)

    assert rc_predict(xp, 10) == GPR_ERR_STATE                    # no evaluation yet
    mm.nlml_grad(hp, want_g=False)
    assert rc_predict(xp, 10) == GPR_ERR_STATE                    # loss-only evaluation: no inverse
    mm.update_cache(hp)
    assert rc_predict(xp, 10) == 0
    assert rc_predict(None, 10) == GPR_ERR_ARG
    assert rc_predict(xp, 0) == GPR_ERR_ARG
    assert rc_predict(xp, 10, same=1) == GPR_ERR_ARG              # same_x needs M == N
    assert L.gpr_mgpu_predict(mm.handle, _ffi.dptr(xp), 10, 0, None, None, None) == GPR_ERR_ARG
    with pytest.raises(gpr.PosDefException):
        mm.update_cache(hp, eps=-10.0)                            # K - 10 I is not positive definite
    assert rc_predict(xp, 10) == GPR_ERR_STATE                    # failed factorization
    mm.update_cache(hp)
    assert rc_predict(xp, 10) == 0
    mm.close(); mc.close()


def test_mgpu_predict_python_mirror_end_to_end(gpr):
    """A few L-BFGS steps of log_loss_grad! on a MultiGPUGradCache, then predict at the result through MultiGPUPredictCache:
    the same as the single-GPU caches at the same hyper-parameters."""
    import scipy.optimize as so
    cov = (o.SE, o.NOISE)
    x, y, hp0, rng = problem(cov, 800, 3, 1, 21)
    md = gpr.GPRModel(to_gpr_cov(gpr, cov), hp0, x, y)
    ll = gpr.MarginalLikelihood()
    tc = gpr.MultiGPUGradCache(md, devices=_devices(3), nb=128)

    def fun(v):
        G = np.empty_like(v)
        return gpr.log_loss_grad_(ll, True, G, v, md, tc), G

    res = so.minimize(fun, np.log(hp0), jac=True, method="L-BFGS-B", options={"maxiter": 5})
    tc.close()
    hp = np.exp(res.x)
    md = gpr.GPRModel(to_gpr_cov(gpr, cov), hp, x, y)
    xp = rng.random((3, 300))
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(3), nb=128)
    gpr.update_cache_(pc, md)
    mu, var, Sf = predict_all(pc, md, xp)
    pc.close()
    mu_s, S_s = gpr.predict(md, xp)
    _, Sd_s = gpr.predict(md, xp, diagonal_var=True)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    prior = float(np.sum(hp[[0, -1]] ** 2))
    assert mean_err(mu, mu_s, y) <= ctol(TOL_MU, cond)
    assert np.abs(var - Sd_s.diag).max() <= ctol(TOL_VAR, cond) * prior
    assert np.abs(Sf - S_s).max() <= ctol(TOL_VAR, cond) * prior
