"""Box integration on the block-cyclic multi-GPU model (gpr_mgpu_integrate).  The GPU tests (pytest -m gpu) cycle the ranks
over the visible GPUs, so a 1-GPU box runs the whole distributed path with several ranks on cuda:0.

Tolerances as in tests/test_mgpu_predict.py: Iout rel 1e-8 against max(|ref|, 1e-8 max|ref|), var abs 1e-8 k2 of the box,
either raised to 10 cond(K) eps where that is larger."""
import re

import numpy as np
import pytest

import gpr_oracle as o
from test_mgpu_predict import _cond_bound, _devices, ctol, mean_err, problem, to_gpr_cov

TOL_I, TOL_VAR = 1e-8, 1e-8
GPR_ERR_ARG, GPR_ERR_STATE, GPR_ERR_UNSUPPORTED = -1, -4, -5


def test_julia_glue_binds_gpr_mgpu_integrate():
    from test_julia_glue import JL, _strip_julia, julia_ccalls
    assert "gpr_mgpu_integrate" in {c[0] for c in julia_ccalls()}
    assert re.search(r"^function integrate_sm100\(s::SM100Multi,", _strip_julia(open(JL).read()), flags=re.M)


def boxes(rng, D, nbox):
    """D x nbox bounds over [-0.2, 1.2]: most boxes reach outside the data's unit cube; with nbox >= 3, box 1 lies far from
    all data (var ~ k2) and box 2 has zero width in dimension 0 (Iout = 0, var = 0)"""
    a = -0.2 + 0.8 * rng.random((D, nbox))
    b = a + 0.05 + 0.6 * rng.random((D, nbox))
    if nbox >= 3:
        a[:, 1], b[:, 1] = 50.0, 51.0
        b[0, 2] = a[0, 2]
    return np.asfortranarray(a), np.asfortranarray(b)


def ref_integrate(mdo, hp, a, b):
    """gpr_oracle.integrate (Cholesky path, src/integrate.jl:103-136) for every column of a, b with one factorization:
    (Iout nbox x ny, var nbox, k2 nbox)"""
    import scipy.linalg as sl
    K = o.kernel(mdo.covar, hp, mdo.x)
    U = sl.cholesky(K, lower=False)
    wt = sl.cho_solve((U, False), mdo.y.reshape(mdo.y.shape[0], -1))
    I, var, k2 = [], [], []
    for i in range(a.shape[1]):
        k1 = o.antideriv(mdo.x, hp, a[:, i], b[:, i])
        tt = sl.solve_triangular(U, k1, trans="T", lower=False)
        k2.append(o.antideriv2(hp, a[:, i], b[:, i]))
        I.append(wt.T @ k1)
        var.append(k2[-1] - float(tt @ tt))
    return np.array(I), np.array(var), np.array(k2)


def check(I, var, I_r, var_r, k2, cond, what):
    """k2 of a zero-width box is 0: its variance is held to 1e-8 of the largest k2 of the batch instead"""
    k2 = np.maximum(k2, 1e-8 * k2.max())
    ei = mean_err(I, I_r, I_r)
    ev = float((np.abs(var - var_r) / k2).max())
    print(f"\n{what}: cond {cond:.1e}, Iout {ei:.1e}, var {ev:.1e} (of k2)")
    assert ei <= ctol(TOL_I, cond)
    assert np.all(np.abs(var - var_r) <= ctol(TOL_VAR, cond) * k2)


# (composition, N, D, ny, nb, G): N = 300 with nb = 128 on 8 ranks leaves ranks without a block; N is no multiple of nb
CASES = [((o.SE, o.NOISE), 300, 3, 1, 128, 8), ((o.SE, o.NOISE), 1000, 2, 3, 256, 2), ((o.SE, o.SE, o.NOISE), 1000, 4, 1, 128, 3),
         ((o.SE, o.SE, o.NOISE), 700, 2, 3, 256, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("cov,N,D,ny,nb,G", CASES)
def test_mgpu_integrate_vs_oracle(gpr, cov, N, D, ny, nb, G):
    x, y, hp, rng = problem(cov, N, D, ny, N + 5 * G + nb)
    ta = 2 if ny > 1 else 1
    mdo = o.GPRModel(cov, hp, x, y, train_axis=ta)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    md = gpr.GPRModel(to_gpr_cov(gpr, cov), hp, x, y, train_axis=ta)
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(G), nb=nb)
    gpr.update_cache_(pc, md)
    # one box through the vector form: gpr_integrate's shapes, and the oracle function itself
    a, b = boxes(rng, D, 1)
    I, var = pc.handle.integrate(a[:, 0], b[:, 0])
    I_o, var_o = o.integrate(mdo, hp, a[:, 0], b[:, 0])
    assert I.shape == (ny,) and var.shape == (1,)
    check(I[None, :], var, I_o[None, :], var_o, np.array([o.antideriv2(hp, a[:, 0], b[:, 0])]), cond, f"{cov} G={G} nbox=1")
    for nbox, tile in ((127, None), (300, 128)):
        if tile:
            pc.mctx.set_option("predict_tile", tile)   # 300 boxes in three tiles
        a, b = boxes(rng, D, nbox)
        I, var = pc.handle.integrate(a, b)
        assert I.shape == (nbox, ny) and var.shape == (nbox,)
        I_r, var_r, k2 = ref_integrate(mdo, hp, a, b)
        check(I, var, I_r, var_r, k2, cond, f"{cov} G={G} nbox={nbox}")
        assert abs(var[1] - k2[1]) <= 1e-9 * k2[1]             # far from all data: nothing is known about the integral
    pc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ozaki", [0, -1])
def test_mgpu_integrate_matches_single_gpu_n8192(gpr, ozaki):
    """Config 2 set A (N = 8192, D = 8, SE + noise) on 4 ranks against gpr_integrate looped over the same 64 boxes, DMMA
    products (ozaki 0) and the automatic route."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("mg2", os.path.join(os.path.dirname(__file__), "golden", "make_golden_config2.py"))
    mg2 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg2)
    x, y, sets = mg2.inputs()
    hp = sets["A"]
    rng = np.random.default_rng(83)
    a, b = boxes(rng, x.shape[0], 64)
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    I_r, var_r = gpr.integrate(md, hp, a, b)
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(4), nb=512)
    pc.mctx.set_option("ozaki", ozaki)
    gpr.update_cache_(pc, md)
    I, var = pc.handle.integrate(a, b)
    pc.close()
    cond = _cond_bound(o.kernel((o.SE, o.NOISE), hp, x), hp[-1] ** 2 + 1e-8)
    k2 = np.array([o.antideriv2(hp, a[:, i], b[:, i]) for i in range(a.shape[1])])
    check(I, var, I_r, var_r, k2, cond, f"N = 8192 on 4 ranks, ozaki {ozaki}")


@pytest.mark.gpu
def test_mgpu_integrate_exact_properties(gpr):
    """On the DMMA pipe: a zero-width box integrates to exactly 0 with variance 0; swapping a_k and b_k negates Iout bit for
    bit and keeps var; transports 0 and 1 agree bit for bit;
    two calls agree; K^-1 is left untouched; every prediction timing slot is used."""
    from gpr_sm100a import _ffi
    x, y, hp, rng = problem((o.SE, o.NOISE), 1000, 3, 1, 9)
    a, b = boxes(rng, 3, 200)
    a2, b2 = a.copy(order="F"), b.copy(order="F")
    a2[1], b2[1] = b[1], a[1]
    outs = []
    for transport in (0, 1):
        mc = _ffi.MultiContext(_devices(3), nb=128, transport=transport)
        mc.set_option("ozaki", 0)
        mm = _ffi.MultiModelHandle(mc, [1, 2], 3, x, y)
        mm.update_cache(hp)
        K0 = mm.fetch(_ffi.FETCH_KINV)
        r1 = mm.integrate(a, b)
        r2 = mm.integrate(a, b)
        assert np.all(r1[0][2] == 0.0) and r1[1][2] == 0.0        # zero width: exactly nothing
        assert all(np.array_equal(u, v) for u, v in zip(r1, r2))
        t = mm.timings()
        assert t["pred_kstar"] > 0 and t["pred_trsm"] > 0 and t["pred_rownorm"] > 0 and t["pred_mean"] > 0, t
        assert np.array_equal(mm.fetch(_ffi.FETCH_KINV), K0)
        s = mm.integrate(a2, b2)
        assert np.array_equal(s[0], -r1[0]) and np.array_equal(s[1], r1[1])
        outs.append(r1)
        mm.close(); mc.close()
    assert all(np.array_equal(u, v) for u, v in zip(outs[0], outs[1]))


@pytest.mark.gpu
def test_mgpu_integrate_agrees_with_quadrature_of_the_posterior_mean(gpr):
    """The integral of the posterior mean over [0, 1]^2 equals 24 x 24 Gauss-Legendre quadrature of gpr_mgpu_predict's mean
    (as test_integrate_agrees_with_quadrature_of_the_posterior_mean on one device)."""
    rng = np.random.default_rng(6)
    dim, n = 2, 400
    x = rng.random((dim, n))
    y = np.sin(x.prod(0)) ** 2
    hp = np.array([1.0, 1.5, 1.5, 0.01])
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(2), nb=128)
    gpr.update_cache_(pc, md)
    I, var = pc.handle.integrate(np.zeros(dim), np.ones(dim))
    xg, wg = np.polynomial.legendre.leggauss(24)
    xg, wg = 0.5 * (xg + 1), 0.5 * wg
    grid = np.asfortranarray(np.stack(np.meshgrid(xg, xg, indexing="ij")).reshape(2, -1))
    pm, _, _ = pc.handle.predict(grid)
    pc.close()
    q = float(np.outer(wg, wg).ravel() @ pm[:, 0])
    print(f"\nIout {I[0]:.15e}, quadrature {q:.15e}, var {var[0]:.3e}")
    assert I[0] == pytest.approx(q, rel=1e-9)
    assert var[0] >= -1e-10


@pytest.mark.gpu
def test_mgpu_integrate_batch_matches_single_boxes(gpr):
    """Box i of a batch (one tile, and tiles of 128) agrees with the nbox = 1 call for box i within the tolerance (not bit for
    bit: the fix-up's split over the columns depends on the tile width)."""
    from gpr_sm100a import _ffi
    cov = (o.SE, o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 900, 3, 1, 13)
    a, b = boxes(rng, 3, 300)
    mc = _ffi.MultiContext(_devices(2), nb=128)
    mm = _ffi.MultiModelHandle(mc, [1, 1, 2], 3, x, y)
    mm.update_cache(hp)
    I, var = mm.integrate(a, b)
    mc.set_option("predict_tile", 128)
    I128, var128 = mm.integrate(a, b)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    k2 = np.array([o.antideriv2(hp, a[:, i], b[:, i]) for i in range(a.shape[1])])
    check(I128, var128, I, var, k2, cond, "tiles of 128 vs one tile")
    idx = [0, 1, 2, 129, 255, 299]
    I1 = np.empty((len(idx), 1)); v1 = np.empty(len(idx))
    for j, i in enumerate(idx):
        Ii, vi = mm.integrate(a[:, i], b[:, i])
        I1[j], v1[j] = Ii, vi[0]
    check(I[idx], var[idx], I1, v1, k2[idx], cond, "batch vs single boxes")
    mm.close(); mc.close()


@pytest.mark.gpu
def test_mgpu_integrate_errors(gpr):
    from gpr_sm100a import _ffi
    x, y, hp, rng = problem((o.SE, o.NOISE), 500, 2, 1, 3)
    a, b = boxes(rng, 2, 4)
    L = _ffi.lib()
    Iout, var = np.empty(4), np.empty(4)
    mc = _ffi.MultiContext(_devices(2), nb=128)
    mm = _ffi.MultiModelHandle(mc, [1, 2], 2, x, y)

    def rc(nbox=4, a_=a, b_=b, I_=Iout, m=None):
        m = m or mm
        return L.gpr_mgpu_integrate(m.handle, nbox, _ffi.dptr(a_), _ffi.dptr(b_), _ffi.dptr(I_), _ffi.dptr(var))

    assert rc() == GPR_ERR_STATE                                   # no evaluation yet
    mm.nlml_grad(hp, want_g=False)
    assert rc() == GPR_ERR_STATE                                   # loss-only evaluation: no inverse
    mm.update_cache(hp)
    assert rc() == 0
    assert rc(a_=None) == GPR_ERR_ARG and rc(b_=None) == GPR_ERR_ARG and rc(I_=None) == GPR_ERR_ARG
    assert rc(nbox=0) == GPR_ERR_ARG
    assert L.gpr_mgpu_integrate(mm.handle, 4, _ffi.dptr(a), _ffi.dptr(b), _ffi.dptr(Iout), None) == 0   # var_out nullable
    with pytest.raises(gpr.PosDefException):
        mm.update_cache(hp, eps=-10.0)                             # K - 10 I is not positive definite
    assert rc() == GPR_ERR_STATE                                   # failed factorization
    mm.update_cache(hp)
    assert rc() == 0
    mm.close(); mc.close()
    # the antiderivative is the SquaredExp one: a WhiteNoise- or Matern-first model is refused, not integrated with it
    for types, P in (([2, 1], 1 + 3), ([3, 2], 3 + 1)):
        mc = _ffi.MultiContext(_devices(2), nb=128)
        m2 = _ffi.MultiModelHandle(mc, types, 2, x, y)
        m2.update_cache(0.3 + rng.random(P))
        assert rc(m=m2) == GPR_ERR_UNSUPPORTED
        m2.close(); mc.close()


@pytest.mark.gpu
def test_mgpu_integrate_python_mirror_end_to_end(gpr):
    """gpr.integrate(..., cache=MultiGPUPredictCache) against the single-device gpr.integrate (one box, a batch; no, scalar
    and vector sample_noise) and, with sample_noise, against the oracle's eigen path (tolerances of
    test_integrate_matches_oracle)."""
    rng = np.random.default_rng(31)
    dim, n, ny = 3, 600, 3
    x = rng.random((dim, n))
    y = rng.random((n, ny))
    hp = np.concatenate([[1.2], 0.8 + 2.0 * rng.random(dim), [0.05]])
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    mdo = o.GPRModel((o.SE, o.NOISE), hp, x, y)
    cond = np.linalg.cond(o.kernel((o.SE, o.NOISE), hp, x))
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(3), nb=128)
    a, b = boxes(rng, dim, 40)
    k2 = np.array([o.antideriv2(hp, a[:, i], b[:, i]) for i in range(a.shape[1])])
    noise = np.array([1e-3, 2e-3, 1e-3])
    for sn in (None, 2e-3, noise):
        I1, v1 = gpr.integrate(md, hp, a[:, 0], b[:, 0], sample_noise=sn, cache=pc)
        I1s, v1s = gpr.integrate(md, hp, a[:, 0], b[:, 0], sample_noise=sn)
        assert I1.shape == I1s.shape and v1.shape == v1s.shape
        IB, vB = gpr.integrate(md, hp, a, b, sample_noise=sn, cache=pc)
        IBs, vBs = gpr.integrate(md, hp, a, b, sample_noise=sn)
        assert IB.shape == IBs.shape == (40, ny) and vB.shape == vBs.shape
        kk = k2 if vB.ndim == 1 else k2[:, None]
        assert mean_err(I1, I1s, I1s) <= ctol(TOL_I, cond) and mean_err(IB, IBs, IBs) <= ctol(TOL_I, cond)
        assert np.all(np.abs(v1 - v1s) <= ctol(TOL_VAR, cond) * k2[0]) and np.all(np.abs(vB - vBs) <= ctol(TOL_VAR, cond) * kk)
        if sn is not None:
            for i in range(0, 40, 13):
                Io, vo = o.integrate(mdo, hp, a[:, i], b[:, i], sn)
                np.testing.assert_allclose(IB[i], Io, rtol=1e-7, atol=1e-8 * np.abs(Io).max())
                np.testing.assert_allclose(vB[i], np.broadcast_to(vo, vB[i].shape), rtol=0, atol=1e-7 * k2[i])
    pc.close()
