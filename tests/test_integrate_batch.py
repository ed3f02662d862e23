"""Box integration of many boxes per call on one GPU (gpr_integrate_batch): one triangular solve per tile of boxes instead of
one trsv per box.

Tolerances as in tests/test_mgpu_integrate.py: Iout rel 1e-8 against max(|ref|, 1e-8 max|ref|), var abs 1e-8 k2 of the box,
either raised to 10 cond(K) eps where that is larger."""
import re

import numpy as np
import pytest

import gpr_oracle as o
from test_mgpu_integrate import boxes, check, ref_integrate
from test_mgpu_predict import _cond_bound, ctol, mean_err, problem, to_gpr_cov

TOL_I, TOL_VAR = 1e-8, 1e-8
GPR_ERR_ARG, GPR_ERR_STATE, GPR_ERR_UNSUPPORTED = -1, -4, -5
TYPES = {o.SE: 1, o.NOISE: 2}


def test_julia_glue_binds_gpr_integrate_batch():
    from test_julia_glue import JL, _strip_julia, julia_ccalls
    assert "gpr_integrate_batch" in {c[0] for c in julia_ccalls()}
    src = _strip_julia(open(JL).read())
    m = re.search(r"^function integrate_sm100\(md::GPRModel,.*?^end$", src, flags=re.M | re.S)
    assert m and re.search(r"Matrix\{Float64\}\(a\)", m.group(0))          # D x nbox bounds are taken as matrices
    once = re.search(r"^function _integrate_once\(h::Handle,.*?^end$", src, flags=re.M | re.S)
    assert once and "a::VecOrMat{Float64}" in once.group(0) and ":gpr_integrate_batch" in once.group(0)


def test_model_handle_integrate_checks_bounds_before_the_device(monkeypatch):
    """(D,) goes to gpr_integrate, (D, nbox) to gpr_integrate_batch; anything else is refused before the library is touched"""
    from gpr_sm100a import _ffi

    class Called(Exception):
        pass

    class FakeLib:
        def __getattr__(self, name):
            raise Called(name)

    class FakeCtx:
        def check(self, rc):
            raise AssertionError("unreachable: the library call raises first")

    monkeypatch.setattr(_ffi, "lib", lambda: FakeLib())
    h = _ffi.ModelHandle.__new__(_ffi.ModelHandle)
    h.D, h.ny, h._h, h.ctx = 3, 1, None, FakeCtx()
    for a, b in ((np.zeros(2), np.ones(2)), (np.zeros(3), np.ones(4)), (np.zeros((3, 2)), np.ones((3, 3))),
                 (np.zeros((2, 4)), np.ones((2, 4))), (np.zeros((3, 0)), np.ones((3, 0))), (np.zeros((3, 2, 1)), np.ones((3, 2, 1))),
                 (np.zeros(3), np.ones((3, 1)))):
        with pytest.raises(_ffi.GPRError, match="integration bounds"):
            h.integrate(a, b)
    with pytest.raises(Called, match="^gpr_integrate$"):
        h.integrate(np.zeros(3), np.ones(3))
    with pytest.raises(Called, match="^gpr_integrate_batch$"):
        h.integrate(np.zeros((3, 5)), np.ones((3, 5)))


def _model(cov, D, x, y, hp, train_axis=1, **options):
    """a fresh context (options set on it) and a model factored at hp, no inverse"""
    from gpr_sm100a import _ffi
    ctx = _ffi.Context(0)
    for k, v in options.items():
        ctx.set_option(k, v)
    m = _ffi.ModelHandle(ctx, [TYPES[c] for c in cov], D, x, y, train_axis)
    m.update_cache(hp)
    return ctx, m


def _k2(hp, a, b):
    return np.array([o.antideriv2(hp, a[:, i], b[:, i]) for i in range(a.shape[1])])


# (composition, N, D, ny): no N is a multiple of 128
CASES = [((o.SE, o.NOISE), 300, 3, 1), ((o.SE, o.NOISE), 700, 2, 3), ((o.SE, o.SE, o.NOISE), 1000, 4, 1),
         ((o.SE, o.SE, o.NOISE), 900, 3, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("cov,N,D,ny", CASES)
def test_integrate_batch_vs_oracle(gpr, cov, N, D, ny):
    x, y, hp, rng = problem(cov, N, D, ny, N + 17)
    ta = 2 if ny > 1 else 1
    mdo = o.GPRModel(cov, hp, x, y, train_axis=ta)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    ctx, m = _model(cov, D, x, y, hp, ta)
    for nbox, tile in ((1, None), (127, None), (300, 128)):
        if tile:
            ctx.set_option("predict_tile", tile)    # 300 boxes in three tiles
        a, b = boxes(rng, D, nbox)
        I, var = m.integrate(a, b)
        assert I.shape == (nbox, ny) and var.shape == (nbox,)
        I_r, var_r, k2 = ref_integrate(mdo, hp, a, b)
        check(I, var, I_r, var_r, k2, cond, f"{cov} ny={ny} nbox={nbox}")
        if nbox >= 3:
            assert abs(var[1] - k2[1]) <= 1e-9 * k2[1]           # far from all data: nothing is known about the integral
            assert np.all(I[2] == 0.0) and var[2] == 0.0         # zero width
    m.close(); ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ozaki", [0, -1])
def test_integrate_batch_matches_gpr_integrate_and_mgpu_n8192(gpr, ozaki):
    """Config 2 set A (N = 8192, D = 8, SE + noise): 64 boxes against gpr_integrate looped over them and against
    gpr_mgpu_integrate with G = 1 on the same model, DMMA products (ozaki 0) and the automatic route."""
    import importlib.util
    import os
    from gpr_sm100a import _ffi
    spec = importlib.util.spec_from_file_location("mg2", os.path.join(os.path.dirname(__file__), "golden", "make_golden_config2.py"))
    mg2 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg2)
    x, y, sets = mg2.inputs()
    hp = sets["A"]
    D = x.shape[0]
    a, b = boxes(np.random.default_rng(83), D, 64)
    ctx, m = _model((o.SE, o.NOISE), D, x, y, hp, ozaki=ozaki)
    I, var = m.integrate(a, b)
    I1, v1 = np.empty((64, 1)), np.empty(64)
    for i in range(64):
        Ii, vi = m.integrate(a[:, i], b[:, i])
        I1[i], v1[i] = Ii, vi[0]
    m.close(); ctx.close()
    mc = _ffi.MultiContext([0], nb=1024)
    mc.set_option("ozaki", ozaki)
    mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
    mm.update_cache(hp)
    Im, vm = mm.integrate(a, b)
    mm.close(); mc.close()
    cond = _cond_bound(o.kernel((o.SE, o.NOISE), hp, x), hp[-1] ** 2 + 1e-8)
    k2 = _k2(hp, a, b)
    check(I, var, I1, v1, k2, cond, f"N = 8192 vs gpr_integrate, ozaki {ozaki}")
    check(I, var, Im, vm, k2, cond, f"N = 8192 vs gpr_mgpu_integrate G = 1, ozaki {ozaki}")


@pytest.mark.gpu
def test_integrate_batch_cache_states(gpr):
    """Works after a loss-only update (no inverse), after a gradient evaluation (inverse formed out of place) and with
    inplace_lauum = 1 (inverse formed in place in its own buffer; U is kept); GPR_ERR_STATE before any factorization and after a
    failed one.  The factor is left untouched."""
    from gpr_sm100a import _ffi
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 600, 3, 1, 21)
    a, b = boxes(rng, 3, 50)
    mdo = o.GPRModel(cov, hp, x, y)
    I_r, var_r, k2 = ref_integrate(mdo, hp, a, b)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    L = _ffi.lib()
    for inplace in (0, 1):
        ctx = _ffi.Context(0)
        ctx.set_option("inplace_lauum", inplace)
        m = _ffi.ModelHandle(ctx, [1, 2], 3, x, y)
        Iout, var = np.empty((50, 1), order="F"), np.empty(50)
        assert L.gpr_integrate_batch(m.handle, 50, _ffi.dptr(a), _ffi.dptr(b), _ffi.dptr(Iout), _ffi.dptr(var)) == GPR_ERR_STATE
        m.update_cache(hp)                                        # MllLossCache: factor, no inverse
        U0 = m.fetch(_ffi.FETCH_U)
        check(*m.integrate(a, b), I_r, var_r, k2, cond, f"loss-only update, inplace_lauum {inplace}")
        assert np.array_equal(m.fetch(_ffi.FETCH_U), U0)
        m.nlml_grad(hp)                                           # gradient: K^-1 next to U
        check(*m.integrate(a, b), I_r, var_r, k2, cond, f"after a gradient, inplace_lauum {inplace}")
        assert np.array_equal(m.fetch(_ffi.FETCH_U), U0)
        with pytest.raises(gpr.PosDefException):
            m.update_cache(hp, eps=-10.0)                         # K - 10 I is not positive definite
        assert L.gpr_integrate_batch(m.handle, 50, _ffi.dptr(a), _ffi.dptr(b), _ffi.dptr(Iout), _ffi.dptr(var)) == GPR_ERR_STATE
        m.close(); ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ny", [1, 3])
def test_integrate_batch_exact_properties(gpr, ny):
    """On the DMMA pipe: a zero-width box integrates to exactly 0 with variance 0; swapping a_k and b_k negates Iout bit for bit
    and keeps var; two calls agree; box i gives the same bits in one tile of 300, in tiles of 128 and as a batch of one (every
    column of the tile is built, solved and reduced on its own, and the products' kernel does not depend on the column count)."""
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 1000, 3, ny, 9)
    a, b = boxes(rng, 3, 300)
    a2, b2 = a.copy(order="F"), b.copy(order="F")
    a2[1], b2[1] = b[1], a[1]
    ctx, m = _model(cov, 3, x, y, hp, 2 if ny > 1 else 1, ozaki=0)
    r1 = m.integrate(a, b)
    r2 = m.integrate(a, b)
    assert np.all(r1[0][2] == 0.0) and r1[1][2] == 0.0
    assert all(np.array_equal(u, v) for u, v in zip(r1, r2))
    s = m.integrate(a2, b2)
    assert np.array_equal(s[0], -r1[0]) and np.array_equal(s[1], r1[1])
    ctx.set_option("predict_tile", 128)
    r128 = m.integrate(a, b)
    assert all(np.array_equal(u, v) for u, v in zip(r1, r128))
    for i in (0, 1, 2, 127, 128, 299):
        Ii, vi = m.integrate(a[:, i:i + 1], b[:, i:i + 1])
        assert np.array_equal(Ii[0], r1[0][i]) and vi[0] == r1[1][i]
    m.close(); ctx.close()


@pytest.mark.gpu
def test_integrate_batch_additivity_and_quadrature(gpr):
    """Iout over a 4 x 4 partition of [0, 1]^2 sums to Iout of the whole square; the whole square equals 24 x 24 Gauss-Legendre
    quadrature of gpr_predict's mean (as test_integrate_agrees_with_quadrature_of_the_posterior_mean for one box)."""
    rng = np.random.default_rng(6)
    dim, n = 2, 400
    x = rng.random((dim, n))
    y = np.sin(x.prod(0)) ** 2
    hp = np.array([1.0, 1.5, 1.5, 0.01])
    ctx, m = _model((o.SE, o.NOISE), dim, x, y, hp)
    e = np.linspace(0.0, 1.0, 5)
    lo = np.asfortranarray(np.stack(np.meshgrid(e[:-1], e[:-1], indexing="ij")).reshape(2, -1))
    hi = np.asfortranarray(np.stack(np.meshgrid(e[1:], e[1:], indexing="ij")).reshape(2, -1))
    Ic, vc = m.integrate(lo, hi)
    Iw, vw = m.integrate(np.zeros((dim, 1)), np.ones((dim, 1)))
    xg, wg = np.polynomial.legendre.leggauss(24)
    xg, wg = 0.5 * (xg + 1), 0.5 * wg
    grid = np.asfortranarray(np.stack(np.meshgrid(xg, xg, indexing="ij")).reshape(2, -1))
    pm, _, _ = m.predict(grid)
    m.close(); ctx.close()
    q = float(np.outer(wg, wg).ravel() @ pm[:, 0])
    print(f"\nIout {Iw[0, 0]:.15e}, sum over cells {Ic[:, 0].sum():.15e}, quadrature {q:.15e}")
    assert abs(Ic[:, 0].sum() - Iw[0, 0]) <= 1e-12 * abs(Iw[0, 0])
    assert Iw[0, 0] == pytest.approx(q, rel=1e-9)
    assert vw[0] >= -1e-10 and np.all(vc >= -1e-10)


@pytest.mark.gpu
def test_integrate_batch_one_pass_and_timings(gpr):
    """With the default tile, 300 boxes cost the launches of one box; a call with variance uses every prediction slot."""
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 800, 3, 1, 4)
    a, b = boxes(rng, 3, 300)
    ctx, m = _model(cov, 3, x, y, hp)
    m.integrate(a, b)                                             # workspaces
    l0 = ctx.launch_count()
    m.integrate(a[:, :1], b[:, :1])
    one = ctx.launch_count() - l0
    l0 = ctx.launch_count()
    m.integrate(a, b)
    assert ctx.launch_count() - l0 == one
    t = m.timings()
    assert t["pred_kstar"] > 0 and t["pred_mean"] > 0 and t["pred_trsm"] > 0 and t["pred_rownorm"] > 0, t
    m.close(); ctx.close()


@pytest.mark.gpu
def test_integrate_batch_errors(gpr):
    from gpr_sm100a import _ffi
    x, y, hp, rng = problem((o.SE, o.NOISE), 500, 2, 1, 3)
    a, b = boxes(rng, 2, 4)
    L = _ffi.lib()
    Iout, var = np.empty(4), np.empty(4)
    ctx, m = _model((o.SE, o.NOISE), 2, x, y, hp)

    def rc(nbox=4, a_=a, b_=b, I_=Iout, v_=var, h=None):
        return L.gpr_integrate_batch((h or m).handle, nbox, _ffi.dptr(a_), _ffi.dptr(b_), _ffi.dptr(I_), _ffi.dptr(v_))

    assert rc() == 0
    assert rc(a_=None) == GPR_ERR_ARG and rc(b_=None) == GPR_ERR_ARG and rc(I_=None) == GPR_ERR_ARG
    assert rc(nbox=0) == GPR_ERR_ARG
    I2 = np.empty(4)
    assert rc(I_=I2, v_=None) == 0 and np.array_equal(I2, Iout)   # var_out nullable
    m.close()
    m2 = _ffi.ModelHandle(ctx, [2, 1], 2, x, y)                    # WhiteNoise first: no SquaredExp antiderivative
    m2.update_cache(0.3 + rng.random(1 + 3))
    assert rc(h=m2) == GPR_ERR_UNSUPPORTED
    m2.close(); ctx.close()


@pytest.mark.gpu
def test_integrate_batch_python_mirror_end_to_end(gpr):
    """gpr.integrate(md, hp, A, B, sample_noise=...) for no, scalar and vector noise: the shapes of the one-box form stacked,
    the values of per-box calls, and for a few boxes the oracle's eigen path (tolerances of test_integrate_matches_oracle)."""
    rng = np.random.default_rng(41)
    dim, n, ny, nbox = 3, 500, 3, 30
    x = rng.random((dim, n))
    y = rng.random((n, ny))
    hp = np.concatenate([[1.2], 0.8 + 2.0 * rng.random(dim), [0.05]])
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    mdo = o.GPRModel((o.SE, o.NOISE), hp, x, y)
    cond = np.linalg.cond(o.kernel((o.SE, o.NOISE), hp, x))
    a, b = boxes(rng, dim, nbox)
    k2 = _k2(hp, a, b)
    for sn in (None, 2e-3, np.array([1e-3, 2e-3, 1e-3])):
        IB, vB = gpr.integrate(md, hp, a, b, sample_noise=sn)
        one = [gpr.integrate(md, hp, a[:, i], b[:, i], sample_noise=sn) for i in range(nbox)]
        I1 = np.stack([r[0] for r in one])
        v1 = np.concatenate([r[1] for r in one]) if sn is None else np.stack([r[1] for r in one])
        assert IB.shape == I1.shape == (nbox, ny) and vB.shape == v1.shape
        kk = k2 if vB.ndim == 1 else k2[:, None]
        assert mean_err(IB, I1, I1) <= ctol(TOL_I, cond)
        assert np.all(np.abs(vB - v1) <= ctol(TOL_VAR, cond) * kk)
        for i in range(0, nbox, 11):
            Io, vo = o.integrate(mdo, hp, a[:, i], b[:, i], sn)
            np.testing.assert_allclose(IB[i], Io, rtol=1e-7, atol=1e-8 * np.abs(Io).max())
            vi = np.atleast_1d(vB[i])                             # (1,) without sample_noise, (ny,) with it
            np.testing.assert_allclose(vi, np.broadcast_to(vo, vi.shape), rtol=0, atol=1e-7 * k2[i])
