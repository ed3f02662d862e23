"""GPU parity tests (pytest -m gpu): the CUDA path, called through the C ABI via the mirrored host API, against
(1) the committed golden fixtures, (2) the CPU oracle on the same seeded inputs, (3) the reference's own
identity tests (ported from /root/reference/test/*.jl), (4) size-independent properties at larger N.

Tolerances (BASELINE.json north_star / SURVEY.md 8d): K entries rel 1e-10; NLML and every gradient component
rel 1e-8 (component error relative to max(|g_i|, 1e-8 |g|)); predictive mean rel 1e-8 (relative to
max(|mu|, 1e-8 |y|_inf)); variance abs 1e-8 * sum sigma^2.  For jitter-only models (no WhiteNoise) the
attainable agreement of two correct FP64 Choleskys is ~cond(K)*eps (SURVEY.md M8), so the tolerance is
max(stated, 10*cond*eps) (round 1 used 50x; the observed errors are 0.02-0.8 cond*eps, and
tests/test_extended_precision.py referees both sides against a longdouble ground truth).
"""
import glob
import os

import numpy as np
import pytest

import gpr_oracle as o

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = sorted(f for f in glob.glob(os.path.join(HERE, "golden", "*.npz")) if not os.path.basename(f).startswith("config"))
EPS = 2.2e-16
TOL_K, TOL_F, TOL_G, TOL_MU, TOL_VAR = 1e-10, 1e-8, 1e-8, 1e-8, 1e-8


def to_gpr_cov(gpr, cov):
    m = {o.SE: gpr.SquaredExp, o.NOISE: gpr.WhiteNoise, o.MATERN52: gpr.Matern52}
    if isinstance(cov, str):
        return m[cov]()
    k = m[cov[0]]()
    for c in cov[1:]:
        k = k + m[c]()
    return k


def case_cov(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg.CASES[name][0]


def ctol(stated, cond):
    return max(stated, 10.0 * cond * EPS)


def grad_err(G, Gref):
    return float((np.abs(G - Gref) / np.maximum(np.abs(Gref), 1e-8 * np.linalg.norm(Gref))).max())


def mean_err(mu, ref, y):
    return float((np.abs(mu - ref) / np.maximum(np.abs(ref), 1e-8 * np.abs(y).max())).max())


# ------------------------------------------------------------------ (1) golden fixtures
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(f)[:-4] for f in GOLDEN])
def test_golden(gpr, path):
    name = os.path.basename(path)[:-4]
    g = np.load(path)
    cov_o = case_cov(name)
    cov = to_gpr_cov(gpr, cov_o)
    x, y, xp, hp = g["x"], g["y"], g["xp"], g["hp"]
    cond = float(g["cond"])
    ta = int(g["train_axis"])
    # covariance.jl / compose_covar.jl
    K = gpr.kernel(cov, hp, x)
    assert np.abs(K / g["K_self"] - 1).max() < TOL_K
    Kc = gpr.kernel(cov, hp, x, xp)
    assert np.abs(Kc / g["K_cross"] - 1).max() < TOL_K
    # deriv_covar.jl
    P = len(hp)
    for i in sorted({1, 2, P - 1, P}):
        dK = gpr.grad(cov, i, hp, x)
        ref = g[f"dK_{i}"]
        if isinstance(dK, gpr.UniformScaling):
            assert ref.shape == (1,) and dK.lam == pytest.approx(ref[0], rel=1e-15)
        else:
            assert np.abs(dK - ref).max() <= TOL_K * np.abs(ref).max()
    # cost.jl: update_cache! / loss / grad! and the cache internals of test_loss.jl:46-48
    md = gpr.GPRModel(cov, hp, x, y, train_axis=ta)
    ll = gpr.MarginalLikelihood()
    tc = gpr.MllGradCache(md)
    gpr.update_cache_(tc, hp, md)
    F = gpr.loss(ll, md, tc)
    G = np.empty(P)
    gpr.grad_(G, ll, md, tc)
    assert abs(F - g["F"]) <= ctol(TOL_F, cond) * abs(g["F"])
    assert grad_err(G, g["G"]) <= ctol(TOL_G, cond)
    U = tc.kchol_base
    assert np.abs(np.triu(U) - np.triu(g["U"])).max() <= ctol(1e-10, cond) * np.abs(g["U"]).max()
    assert np.abs(np.tril(U, -1) / np.tril(g["K_self"], -1).clip(1e-300) - np.tril(np.ones_like(U), -1)).max() < TOL_K  # strict lower keeps K
    assert np.abs(tc.alpha - g["alpha"]).max() <= ctol(TOL_F, cond) * np.abs(g["alpha"]).max()
    assert np.abs(tc.K_inv - g["Kinv"]).max() <= ctol(TOL_F, cond) * np.abs(g["Kinv"]).max()
    Glog = np.empty(P)
    Fl = gpr.log_loss_grad_(ll, True, Glog, np.log(hp), md, tc)
    assert abs(Fl - g["F"]) <= ctol(TOL_F, cond) * abs(g["F"])
    assert grad_err(Glog, g["G_log"]) <= ctol(TOL_G, cond)
    tc.close()
    # predict.jl
    pc = gpr.GPRPredictCache(md, xp)
    gpr.update_cache_(pc, md)
    M = xp.shape[1]
    mu = np.empty(g["pred_mean"].shape)
    Sd = gpr.Diagonal(np.empty(M))
    gpr.predict_(mu, Sd, md, xp, pc)
    assert mean_err(mu, g["pred_mean"], y) <= ctol(TOL_MU, cond)
    prior = float(np.sum([h[0] ** 2 for h in o.split(hp, [o.dim_hp(k, x.shape[0]) for k in o.as_list(cov_o)])]))
    assert np.abs(Sd.diag - g["pred_var"]).max() <= ctol(TOL_VAR, cond) * prior
    mu2 = np.empty(g["pred_mean"].shape)
    Sf = np.empty((M, M))
    gpr.predict_(mu2, Sf, md, xp, pc)
    assert np.abs(Sf - g["pred_cov"]).max() <= ctol(TOL_VAR, cond) * prior
    assert np.abs(pc.wt - g["wt"]).max() <= ctol(TOL_F, cond) * np.abs(g["wt"]).max()
    mus = np.empty(g["pred_mean_same_x"].shape)
    gpr.predict_mean_(mus, md, md.x, pc)                    # xp === md.x -> jitter on K* too (SURVEY A.2)
    assert mean_err(mus, g["pred_mean_same_x"], y) <= ctol(TOL_MU, cond)
    pc.close()
    # split_kernel.jl / split_predict.jl
    if "split_A" in g.files:
        xe, xq = g["xe"], g["xq"]
        cm = gpr.Cmap(np.add, xe, xq)
        sk = gpr.kernel(cov, hp, cm, x)
        for got, ref in ((sk.A, g["split_A"]), (sk.B, g["split_B"]), (sk.C, g["split_C"])):
            assert np.abs(got / ref - 1).max() < TOL_K
        spc = gpr.GPRSplitPredictCache(md, cm)
        gpr.update_cache_(spc, md)
        smu = np.empty((xe.shape[1], xq.shape[1]))
        sS = gpr.Diagonal(np.empty(smu.size))
        gpr.predict_(smu, sS, md, cm, spc)
        assert mean_err(smu, g["split_mean"], y) <= ctol(TOL_MU, cond)
        assert np.abs(sS.diag - g["split_var"]).max() <= ctol(TOL_VAR, cond) * prior
        spc.var_range = (1, xe.shape[1])
        gpr.predict_(smu, sS, md, cm, spc)
        assert np.abs(sS.diag - g["split_var_all"]).max() <= ctol(TOL_VAR, cond) * prior
        spc.close()


# ------------------------------------------------------------------ (2)+(3) reference tests, against the oracle
@pytest.mark.parametrize("n,dim", [(100, 1), (200, 4), (300, 7)])
def test_covariance_reference_suite(gpr, n, dim):
    """test/test_covariance.jl:13-105"""
    rng = np.random.default_rng(n + dim)
    x, xp = rng.random((dim, n)), rng.random((dim, 2 * n))
    SE, WN = gpr.SquaredExp(), gpr.WhiteNoise()
    hp = rng.random(dim + 1)
    Kxx, Kxp = gpr.kernel(SE, hp, x), gpr.kernel(SE, hp, x, xp)
    assert np.array_equal(Kxx, Kxx.T)
    assert np.all(np.linalg.eigvalsh(Kxx) > 0)
    assert Kxx.shape == (n, n) and Kxp.shape == (n, 2 * n)
    assert np.abs(Kxx / o.kernel(o.SE, hp, x) - 1).max() < TOL_K
    assert np.abs(Kxp / o.kernel(o.SE, hp, x, xp) - 1).max() < TOL_K
    I = np.eye(n)
    for cov, cov_o in ((SE + WN, (o.SE, o.NOISE)), (SE + SE, (o.SE, o.SE)), (SE + SE + WN, (o.SE, o.SE, o.NOISE)),
                       (WN + SE, (o.NOISE, o.SE)), (SE + WN + SE, (o.SE, o.NOISE, o.SE))):
        hps = rng.random(gpr.dim_hp(cov, dim))
        Ks, Kc = gpr.kernel(cov, hps, x), gpr.kernel(cov, hps, x, xp)
        assert np.abs(Ks / o.kernel(cov_o, hps, x) - 1).max() < TOL_K
        assert np.abs(Kc / o.kernel(cov_o, hps, x, xp) - 1).max() < TOL_K
        # composition identity through the library itself
        parts = gpr.split(hps, [gpr.dim_hp(k, dim) for k in cov.kernels])
        acc, accc = np.zeros((n, n)), np.zeros((n, 2 * n))
        for k, h in zip(cov.kernels, parts):
            if isinstance(k, gpr.WhiteNoise):
                acc += h[0] ** 2 * I
            else:
                acc += gpr.kernel(SE, h, x)
                accc += gpr.kernel(SE, h, x, xp)
        np.testing.assert_allclose(Ks, acc, rtol=1.5e-8)
        np.testing.assert_allclose(Kc, accc, rtol=1.5e-8)
    # :84-87 derivative vs forward difference (all i, not only i = dim)
    K0 = gpr.kernel(SE, hp, x)
    for i in range(1, dim + 2):
        hpe = hp.copy()
        hpe[i - 1] += 1e-7
        fd = (gpr.kernel(SE, hpe, x) - K0) / 1e-7
        np.testing.assert_allclose(gpr.grad(SE, i, hp, x), fd, atol=1e-3)
    # :89-105 composed index map
    x2 = rng.random((2, 100))
    cov = SE + WN + SE
    hp7 = rng.random(7)
    hs = gpr.split(hp7, [3, 1, 3])
    for i, (c, li) in {1: (0, 1), 2: (0, 2), 3: (0, 3), 5: (2, 1), 6: (2, 2), 7: (2, 3)}.items():
        np.testing.assert_allclose(gpr.grad(cov, i, hp7, x2), gpr.grad(SE, li, hs[c], x2), rtol=1.5e-8)
    assert gpr.grad(cov, 4, hp7, x2).lam == pytest.approx(2 * hs[1][0])


@pytest.mark.parametrize("dim,shift,scale", [(2, 0.0, 40.0), (8, 1000.0, 1.0), (4, 0.0, 6.0), (16, -50.0, 2.0)])
def test_gram_form_and_table_exp_accuracy(gpr, ctx, dim, shift, scale):
    """The TMA-fed Gram-form build (csrc/kbuild_tma.cuh: d = |a|^2 + |b|^2 - 2 a.b on the DMMA pipe, centred; table-driven
    exp, csrc/fastexp.cuh) against the oracle's direct difference + libm exp (src/covariance.jl:72-95) where they are most
    exposed: distances up to the underflow threshold of exp (K entries down to 1e-300), inputs far from the origin
    (cancellation in the Gram form), and against the direct-difference kernel of the library itself (option
    kbuild_gram = 0).  Tolerance: the stated 1e-10 relative on every K entry that is not subnormal."""
    rng = np.random.default_rng(dim)
    n, m = 300, 200
    x, xp = shift + scale * rng.random((dim, n)), shift + scale * rng.random((dim, m))
    SE, WN = gpr.SquaredExp(), gpr.WhiteNoise()
    hp = np.concatenate([[1.3], 0.5 + rng.random(dim), [0.7], 0.2 + rng.random(dim), [0.1]])
    cov, cov_o = SE + SE + WN, (o.SE, o.SE, o.NOISE)
    Kref, Kcref = o.kernel(cov_o, hp, x), o.kernel(cov_o, hp, x, xp)
    for flag in (1, 0):
        ctx.set_option("kbuild_gram", flag)
        try:
            Ks, Kc = gpr.kernel(cov, hp, x), gpr.kernel(cov, hp, x, xp)
        finally:
            ctx.set_option("kbuild_gram", 1)
        for got, ref in ((Ks, Kref), (Kc, Kcref)):
            big = ref > 1e-300
            err = np.abs(got[big] / ref[big] - 1).max()
            print(f"\nD={dim} shift={shift} scale={scale} gram={flag}: max rel err {err:.2e} over {big.sum()} entries, min K {ref[big].min():.1e}")
            assert err < TOL_K
            assert np.all(np.abs(got[~big]) <= 1e-299)
        assert np.array_equal(Ks, Ks.T)                      # symmetric to the last bit
        assert np.all(np.diag(Ks) == np.diag(Kref))           # d_ii = 0 exactly -> sigma^2 (+ eps, + noise) exactly


@pytest.mark.parametrize("n,dim,ny", [(10, 2, 1), (20, 5, 1), (100, 2, 1), (100, 5, 5), (300, 3, 10)])
def test_loss_reference_suite(gpr, n, dim, ny):
    """test/test_loss.jl:21-97"""
    rng = np.random.default_rng(n * 31 + dim + ny)
    x = rng.random((dim, n))
    y1 = np.sin(x).sum(0)
    if ny == 1:
        y, ta = y1, 1
    else:
        y = np.stack([rng.random() * y1 for _ in range(ny)], axis=1)
        ta = int(rng.integers(1, ny + 1))
    cov, cov_o = gpr.SquaredExp() + gpr.WhiteNoise(), (o.SE, o.NOISE)
    hp = 0.05 + rng.random(dim + 2)
    md = gpr.GPRModel(cov, hp, x, y, train_axis=ta)
    ll = gpr.MarginalLikelihood()
    yt = gpr.get_sample(md)
    mdo = o.GPRModel(cov_o, hp, x, y, train_axis=ta)
    tco = o.MllGradCache(mdo)
    Fo, Go = o.loss_grad(hp, mdo, tco)
    cond = np.linalg.cond(o.kernel(cov_o, hp, x))
    assert gpr.loss(ll, cov, hp, x, yt) == pytest.approx(gpr.loss(ll, hp, md), rel=1.5e-8)      # :35 functional == cached
    assert gpr.loss(ll, hp, md) == pytest.approx(Fo, rel=ctol(TOL_F, cond))
    DL1 = gpr.grad(ll, hp, md)
    assert grad_err(DL1, Go) <= ctol(TOL_G, cond)
    tc = gpr.MllGradCache(md)
    gpr.update_cache_(tc, hp, md)
    assert np.abs(tc.kchol_base - tco.kchol_base).max() <= ctol(1e-10, cond) * np.abs(tco.kchol_base).max()   # :46
    assert np.abs(tc.alpha - tco.alpha).max() <= ctol(TOL_F, cond) * np.abs(tco.alpha).max()                  # :47
    assert np.abs(tc.K_inv - tco.Kinv).max() <= ctol(TOL_F, cond) * np.abs(tco.Kinv).max()                    # :48
    for i in range(len(hp)):                                                                                  # :50-55
        hpe = hp.copy()
        hpe[i] += 1e-6
        fd = (gpr.loss(ll, hpe, md, tc) - gpr.loss(ll, hp, md, tc)) / 1e-6
        assert DL1[i] == pytest.approx(fd, rel=2e-3, abs=1e-3 * max(1.0, abs(fd)))
    tc.close()


def test_nlml_known_answer_diagonal(gpr):
    """test/test_loss.jl:1-11 through the device: an SE kernel with a huge inverse length scale is diagonal,
    K = (sigma^2 + eps + sigma_n^2) I, so NLML has the closed form of the reference's known-answer test."""
    rng = np.random.default_rng(3)
    n = 200
    x = np.arange(n, dtype=np.float64)[None, :]
    y = rng.random(n)
    hp = np.array([0.8, 50.0, 0.3])
    d = 0.8 ** 2 + 1e-8 + 0.3 ** 2
    mle = 0.5 * (np.dot(y, y) / d + n * np.log(d) + n * np.log(2 * np.pi))
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    assert gpr.loss(gpr.MarginalLikelihood(), hp, md) == pytest.approx(mle, rel=1e-13)


def test_not_positive_definite_raises(gpr):
    """cholesky!(...; check=true) throws PosDefException (src/cost.jl:77)"""
    x = np.zeros((1, 300))           # identical points, no jitter -> singular K
    y = np.ones(300)
    md = gpr.GPRModel(gpr.SquaredExp(), np.array([1.0, 1.0]), x, y)
    tc = gpr.MllLossCache(md)
    with pytest.raises(gpr.PosDefException) as ei:
        gpr.update_cache_(tc, md.params, md, ϵ=0.0)
    assert 1 <= ei.value.info <= 300
    # gradient cache: the factorization status is read once AFTER the inverse has been enqueued (no host round trip between potrf
    # and the inverse) -- the failure must surface the same way, and the cache must recover on the next valid evaluation
    tg = gpr.MllGradCache(md)
    with pytest.raises(gpr.PosDefException) as eg:
        gpr.update_cache_(tg, md.params, md, ϵ=0.0)
    assert eg.value.info == ei.value.info
    gpr.update_cache_(tg, md.params, md, ϵ=1.0)                  # K = 1 1^T + I: positive definite
    gpr.update_cache_(tc, md.params, md, ϵ=1.0)
    ll = gpr.MarginalLikelihood()
    Fg, Fl = gpr.loss(ll, md, tg), gpr.loss(ll, md, tc)            # loss(cost, md, tc): from the cache as it stands (src/cost.jl:113-117)
    # closed form: eigenvalues 301 (once) and 1; y = 1: y^T K^-1 y = 300 / 301
    Fref = 0.5 * (300.0 / 301.0 + np.log(301.0) + 300 * np.log(2 * np.pi))
    assert Fg == pytest.approx(Fref, rel=1e-12) and Fl == pytest.approx(Fref, rel=1e-12)
    tg.close()
    tc.close()


@pytest.mark.parametrize("n,npred,dim", [(100, 100, 1), (200, 500, 2), (500, 200, 5)])
def test_predict_reference_suite(gpr, n, npred, dim):
    """test/test_models.jl:1-48"""
    rng = np.random.default_rng(n + npred + dim)
    x, xp = rng.random((dim, n)), rng.random((dim, npred))
    y = np.sin(x.sum(0)) ** 2
    SE, WN = gpr.SquaredExp(), gpr.WhiteNoise()
    md2 = gpr.GPRModel(SE + SE, 0.2 + rng.random(2 * (dim + 1)), x, y)
    np.testing.assert_allclose(gpr.predict_mean(md2, x), y, rtol=1e-5, atol=1e-5)        # :19 interpolation
    _, S = gpr.predict(md2, x)
    assert np.abs(S).max() < 1e-5                                                         # :24
    hp3 = rng.random(dim + 2)
    hp3[-1] = 1e-5
    md3 = gpr.GPRModel(SE + WN, hp3, x, y)
    mu3 = gpr.predict_mean(md3, x)
    # :28 interpolation property; the reference asserts rtol 1e-3 on rand() hyper-parameters (statistical), so the
    # hard check here is agreement with the oracle on the same inputs and a looser interpolation bound
    np.testing.assert_allclose(mu3, y, rtol=1e-2, atol=1e-2)
    mdo3 = o.GPRModel((o.SE, o.NOISE), hp3, x, y)
    cond3 = np.linalg.cond(o.kernel((o.SE, o.NOISE), hp3, x))
    # sigma_n = 1e-5: cond(K) ~ 1e9-1e10, agreement of two correct Choleskys is ~1e3 * cond * eps at best
    assert mean_err(mu3, o.predict_mean(mdo3, x, same=True), y) <= max(TOL_MU, 2000.0 * cond3 * EPS)
    md = gpr.GPRModel(SE + WN, 0.1 + rng.random(dim + 2), x, y)
    yp, Sf = gpr.predict(md, xp)
    yd, Sd = gpr.predict(md, xp, diagonal_var=True)
    np.testing.assert_allclose(np.diag(Sf), Sd.diag, atol=1e-5)                           # :41
    mdo = o.GPRModel((o.SE, o.NOISE), md.params, x, y)
    cond = np.linalg.cond(o.kernel((o.SE, o.NOISE), md.params, x))
    mu_o, var_o = o.predict(mdo, xp, diagonal_var=True)
    assert mean_err(yp, mu_o, y) <= ctol(TOL_MU, cond) and mean_err(yd, mu_o, y) <= ctol(TOL_MU, cond)
    assert np.abs(Sd.diag - var_o).max() <= ctol(TOL_VAR, cond) * o.prior_diag(mdo)
    md1 = gpr.GPRModel(SE, 0.5 + rng.random(dim + 1), x, y)
    _, Sf = gpr.predict(md1, xp)
    _, Sd = gpr.predict(md1, xp, diagonal_var=True)
    np.testing.assert_allclose(np.diag(Sf), Sd.diag, atol=1e-5)                           # :47


@pytest.mark.parametrize("cov_id", [0, 1, 2, 3])
@pytest.mark.parametrize("dim,n,e,q", [(1, 100, 10, 10), (2, 200, 20, 30), (5, 500, 50, 10)])
def test_split_reference_suite(gpr, cov_id, dim, n, e, q):
    """test/test_split_kernel.jl:1-78"""
    SE, WN = gpr.SquaredExp(), gpr.WhiteNoise()
    cov = [SE, SE + WN, SE + SE, SE + SE + WN][cov_id]
    rng = np.random.default_rng(cov_id * 1000 + n + e + q)
    x, xe, xq = rng.random((dim, n)), rng.random((dim, e)), rng.random((dim, q))
    y = np.sin(x.sum(0)) ** 2
    hp = 0.2 + rng.random(gpr.dim_hp(cov, dim))
    xeq = gpr.Cmap(np.add, xe, xq)
    KK = gpr.kernel(cov, hp, xeq[:, :], x)
    Kxp = gpr.kernel(cov, hp, xeq, x)
    for (ee, qq, s) in ((0, 0, n - 1), (e - 1, q - 1, n - 1), (3, 2, 5)):
        assert Kxp[ee, qq, s] == pytest.approx(KK[qq * e + ee, s], rel=1e-9)               # :36-44
    md = gpr.GPRModel(cov, hp, x, y)
    yp, varp = gpr.predict(md, xeq[:, :], diagonal_var=True)
    yps, varps = gpr.predict(md, xeq, diagonal_var=True)
    np.testing.assert_allclose(yps.reshape(-1, order="F"), yp, rtol=1e-6, atol=1e-8)       # :67-69
    xqe = gpr.Cmap(np.add, xq, xe)
    _, varpt = gpr.predict(md, xqe[:, :], diagonal_var=True)
    np.testing.assert_allclose(varps.diag[:3 * q], varpt.diag[:3 * q], rtol=1e-5, atol=1e-8)   # :75
    assert not np.allclose(varps.diag[:3 * q + 1], varpt.diag[:3 * q + 1], rtol=1e-5, atol=0)  # :76


def test_train_matches_oracle_trajectory(gpr):
    """Config 1 (BASELINE.json): 1-D sin(x)+noise, N=1000, SquaredExp()+WhiteNoise(), hyper-parameter training
    from log-hp0 = ones with the same host optimiser on the CUDA path and on the oracle (src/train.jl:47-56)."""
    import scipy.optimize as so
    rng = np.random.default_rng(1001)
    N = 1000
    x = 10.0 * rng.random((1, N))
    y = np.sin(x[0]) + 0.1 * rng.standard_normal(N)
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), np.ones(3), x, y)
    hp_gpu, res = gpr.train(md, gpr.MarginalLikelihood(), method="L-BFGS-B", options={"gtol": 1e-2, "maxiter": 60})
    mdo = o.GPRModel((o.SE, o.NOISE), np.ones(3), x, y)
    tco = o.MllGradCache(mdo)
    res_o = so.minimize(lambda v: o.log_loss_grad(v, mdo, tco), np.ones(3), jac=True, method="L-BFGS-B",
                        options={"gtol": 1e-2, "maxiter": 60})
    np.testing.assert_allclose(hp_gpu, np.exp(res_o.x), rtol=1e-6)
    assert res.fun == pytest.approx(res_o.fun, rel=1e-9)
    assert 0.05 < hp_gpu[2] < 0.2          # recovers the noise level 0.1


def test_tma_fed_gemm_matches_ldgsts_gemm(gpr):
    """csrc/dgemm_tma.cuh (operand ring filled by cp.async.bulk.tensor + mbarriers, swizzled fragment loads) against
    numpy and against the LDGSTS kernel: plain, accumulate (beta), upper-only and the triangular K-from-N product, and a
    whole factor + inverse with the option on (every T,N product of potrf / trtri_t / lauum_oop_t, incl. batched levels)."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(12)
    ctx = gpr.Context(0)
    try:
        for (M, N, K, flags, beta) in ((128, 64 * 2, 16, 0, 0.0), (256, 384, 48, 0, 0.0), (512, 256, 1040, 0, 0.5), (384, 384, 384, 1, 1.0),
                                       (512, 512, 512, 3, 0.0), (1024, 1152, 2048, 0, -1.0)):
            A = np.asfortranarray(rng.standard_normal((K, M)))
            B = np.asfortranarray(rng.standard_normal((K, N)))
            C0 = np.asfortranarray(rng.standard_normal((M, N)))
            outs = []
            for tma in (0, 1):
                ctx.set_option("gemm_tma", tma)
                C, _ = _ffi.dbg_dgemm(ctx, "T", "N", 0.75, A, B, beta, C0, flags=flags)
                outs.append(C)
            ref = 0.75 * (A.T @ B) + beta * C0
            if flags & 2:      # K-from-N: tile column block J contracts over k >= 128 J only
                ref = beta * C0.copy()
                for J in range(N // 128):
                    ref[:, 128 * J:128 * (J + 1)] += 0.75 * (A[128 * J:, :].T @ B[128 * J:, 128 * J:128 * (J + 1)])
            mask = np.ones((M, N), dtype=bool)
            if flags & 1:
                mask = np.triu(mask)
            assert np.array_equal(outs[0][mask], outs[1][mask]), (M, N, K, flags)          # same arithmetic order -> same bits
            assert np.abs(outs[1] - ref)[mask].max() <= 1e-12 * max(1.0, np.abs(ref).max()) * K ** 0.5
            if flags & 1:
                assert np.array_equal(outs[1][~mask], C0[~mask])                            # below the diagonal untouched
        n = 1536
        X = rng.standard_normal((n, n))
        Kmat = X @ X.T / n + np.eye(n)
        res = []
        for tma in (0, 1):
            ctx.set_option("gemm_tma", tma)
            res.append(_ffi.dbg_factor(ctx, Kmat.copy(order="F"), mode=3)[0])
        assert np.array_equal(np.triu(res[0]), np.triu(res[1]))
        assert np.abs(np.triu(res[1]) - np.triu(np.linalg.inv(Kmat))).max() <= 1e-11 * np.abs(np.linalg.inv(Kmat)).max()
        # tile-mapped forms (block-cyclic multi-GPU drivers) and the Hadamard epilogue (split-predict mean): TMA on vs off
        mats = []
        for tma in (0, 1):
            mc = _ffi.MultiContext([0, 0, 0], nb=256)
            mc.set_option("gemm_tma", tma)
            A, Y, _ = mc.dbg_factor(np.triu(Kmat), rng.standard_normal((n, 2)) * 0 + 1.0, 2)
            mc.close()
            mats.append((A, Y))
        assert np.array_equal(mats[0][0], mats[1][0]) and np.array_equal(mats[0][1], mats[1][1])
    finally:
        ctx.set_option("gemm_tma", 1)
        ctx.close()


def test_ozaki_int8_gemm_is_an_fp64_product(gpr):
    """csrc/ozaki_i8.cuh: C = alpha A^T B + beta C through tcgen05.mma kind::i8 (8 signed 7-bit digits per operand row,
    36 exact integer products in TMEM, FP64 recombination) against a longdouble product.  The error is measured relative to
    |A|^T |B| (the natural scale of a dot product) and compared with numpy's DGEMM on the same data; flags: upper-only and
    the triangular K-from-N product of the inverse."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(99)
    ctx = gpr.Context(0)
    try:
        for (M, N, K, alpha, beta, flags, kind) in ((128, 128, 128, 1.0, 0.0, 0, "g"), (256, 384, 640, -1.0, 1.0, 0, "g"), (512, 512, 4096, 1.0, 0.5, 1, "g"),
                                                    (384, 384, 384, 1.0, 0.0, 3, "tri"), (256, 256, 32768, 1.0, 0.0, 0, "g"), (512, 640, 2048, 1.0, 1.0, 0, "decay")):
            if kind == "tri":      # triangular op(B) with GARBAGE above its diagonal blocks (the Z11 operand of trtri_t)
                A = np.tril(rng.standard_normal((K, M)))
                B = A.copy()
                for J in range(M // 128):
                    B[:128 * J, 128 * J:128 * (J + 1)] = 1e30
            elif kind == "decay":
                A = rng.standard_normal((K, M)) * np.exp(-4 * rng.random((K, M)))
                B = rng.standard_normal((K, N)) * np.exp(-4 * rng.random((K, N)))
            else:
                A, B = rng.standard_normal((K, M)), rng.standard_normal((K, N))
            A, B = np.asfortranarray(A), np.asfortranarray(B)
            C0 = np.asfortranarray(rng.standard_normal((M, N)))
            C, _ = _ffi.dbg_ozaki_dgemm(ctx, alpha, A, B, beta, C0, S=8, flags=flags)
            Ae, Be = A.copy(), np.tril(B) if kind == "tri" else B.copy()
            if flags & 2:          # column block J contracts over k >= 128 J only
                ref = beta * C0.astype(np.longdouble)
                den = np.zeros((M, N))
                for J in range(N // 128):
                    sl = slice(128 * J, 128 * (J + 1))
                    ref[:, sl] += alpha * (Ae[128 * J:, :].astype(np.longdouble).T @ Be[128 * J:, sl].astype(np.longdouble))
                    den[:, sl] = np.abs(Ae[128 * J:, :]).T @ np.abs(Be[128 * J:, sl])
            else:
                ref = alpha * (Ae.astype(np.longdouble).T @ Be.astype(np.longdouble)) + beta * C0
                den = np.abs(Ae).T @ np.abs(Be)
            mask = np.triu(np.ones((M, N), dtype=bool)) if flags & 1 else np.ones((M, N), dtype=bool)
            err = float(np.max((np.abs(C - ref) / (den + 1e-300))[mask]))
            print(f"\nozaki {M}x{N}x{K} flags={flags} {kind}: max err / (|A|^T|B|) = {err:.2e}")
            # norm-wise accuracy: entries formed by few / small terms under a large row maximum (triangular corner, decaying
            # magnitudes) carry an error relative to the row maxima, not to their own terms
            assert err < (4e-16 if kind == "g" else 5e-14)
            if flags & 1:
                assert np.array_equal(C[~mask], C0[~mask])
    finally:
        ctx.close()


def test_ozaki_nine_digit_two_window_product(gpr):
    """The W^T W product of the inverse takes NINE digits (csrc/ozaki_i8.cuh: 45 integer products in two diagonal windows,
    d = 6..10 with 128 x 96 tiles | d = 2..5): on operands whose entries span many orders of magnitude under one scale per column
    it must be at least 16x closer to the exact product than the 8-digit form, and honour upper-only / K-from-N (lauum_oop_t's
    flags) on a size that is no multiple of the 96-wide tiles."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(77)
    ctx = gpr.Context(0)
    try:
        K, M = 1024, 640
        A = np.asfortranarray(rng.standard_normal((K, M)) * np.exp(rng.uniform(-14, 0, (K, M))))
        ref = (A.astype(np.longdouble).T @ A.astype(np.longdouble))
        den = np.abs(A).T @ np.abs(A)
        err = {}
        out = {}
        for S in (8, 9):
            out[S], _ = _ffi.dbg_ozaki_dgemm(ctx, 1.0, A, A, 0.0, np.zeros((M, M)), S=S, flags=0)
            err[S] = float(np.max(np.abs(out[S] - ref) / den))
        print(f"\nW^T W with 6 decades inside a column: err/(|A|^T|A|) 8 digits {err[8]:.2e}, 9 digits {err[9]:.2e}")
        assert err[9] < 2e-15
        assert err[9] * 16 <= err[8] or err[8] < 1e-15
        # lauum_oop_t's form: lower-triangular operand (garbage above the diagonal blocks), upper triangle of C only
        Kt = 640
        L = np.tril(rng.standard_normal((Kt, Kt))) + 4 * np.eye(Kt)
        G = L.copy()
        for J in range(Kt // 128):
            G[:128 * J, 128 * J:128 * (J + 1)] = 1e30
        G = np.asfortranarray(G)
        reft = L.astype(np.longdouble).T @ L.astype(np.longdouble)
        dent = np.abs(L).T @ np.abs(L)
        C0 = np.asfortranarray(rng.standard_normal((Kt, Kt)))
        Cm, _ = _ffi.dbg_ozaki_dgemm(ctx, 1.0, np.asfortranarray(L), G, 0.0, C0, S=9, flags=3)      # separate operands: only op(B) is masked
        up = np.triu(np.ones((Kt, Kt), dtype=bool))
        e = float(np.max((np.abs(Cm - reft) / dent)[up]))
        print(f"L^T L, K-from-N + upper-only: err {e:.2e}")
        assert e < 2e-15
        assert np.array_equal(Cm[~up], C0[~up])
    finally:
        ctx.close()


def test_ozaki_rejects_retired_forms(gpr):
    """Forms of the INT8 product that no kernel serves fail cleanly: option names of retired variants are unknown to the
    context, and launch_ozaki_dgemm refuses nine digits with the tile-mapped or skip-tile forms, the two-window 8-digit form
    with the tile-mapped forms, and flags it does not know.  The context stays usable afterwards."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(5)
    ctx = gpr.Context(0)
    try:
        for name in ("ozaki_mc", "ozaki_windows", "ozaki_lauum_map"):
            with pytest.raises(_ffi.GPRError, match="unknown option"):
                ctx.set_option(name, 0)
        A = np.asfortranarray(rng.standard_normal((256, 256)))
        C0 = np.zeros((256, 256), order="F")
        for S, fl in ((9, 8), (9, 16), (9, 32), (9, 64), (9, 1 | 64), (8, 512 | 8), (8, 512 | 16), (8, 1024), (8, 4096), (8, 8192),
                      (9, 1024), (9, 4096), (8, 512 | 8192), (8, 32)):
            with pytest.raises(_ffi.GPRError):
                _ffi.dbg_ozaki_dgemm(ctx, 1.0, A, A, 0.0, C0, S=S, flags=fl)
        C, _ = _ffi.dbg_ozaki_dgemm(ctx, 1.0, A, A, 0.0, C0, S=9, flags=3)
        assert np.all(np.isfinite(C))
    finally:
        ctx.close()


def test_ozaki_route_keeps_nlml_parity(gpr):
    """The INT8-tensor-core route of the blocked factorization (ctx option "ozaki" = 8 digits for potrf, trtri and the
    prediction solves; "ozaki_lauum" = 9 digits for the W^T W product of the inverse) against the oracle on a model large
    enough that its top-level products are routed there (ozaki_min = 512): same tolerances as the DMMA path
    (src/cost.jl:96-127, src/predict.jl:83-95)."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(4242)
    D, N = 8, 4096
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.5 * np.ones(D), [0.5], 2.0 * np.ones(D), [0.1]])
    xp = np.asfortranarray(rng.random((D, 2048)))
    mdo = o.GPRModel((o.SE, o.SE, o.NOISE), hp, x, y)
    Fo, Go = o.loss_grad(hp, mdo)
    mu_o, var_o = o.predict(mdo, xp, diagonal_var=True)
    xe_s, xq_s = np.asfortranarray(0.5 * rng.random((D, 512))), np.asfortranarray(0.5 * rng.random((D, 512)))
    mu_split_o = {e: o.predict(mdo, xe_s[:, e:e + 1] + xq_s, diagonal_var=True)[0] for e in (0, 255, 511)}     # rows of the sum grid
    ctx = gpr.Context(0)
    try:
        res = {}
        for oz in (0, 8):
            ctx.set_option("ozaki", oz)
            ctx.set_option("ozaki_min", 512)
            mh = _ffi.ModelHandle(ctx, [1, 1, 2], D, np.asfortranarray(x), y)
            l0 = ctx.launch_count()
            F, G = mh.nlml_grad(hp)
            mu, var, _ = mh.predict(xp, want_var=True)
            # split-predict mean (src/split_predict.jl:10-19): its T,N products with the Hadamard epilogue take the same route
            ms_, _ = mh.split_predict(xe_s, xq_s, var_range=None, want_var=False)
            split_err = max(mean_err(ms_[e, :], mu_split_o[e], y) for e in mu_split_o)
            res[oz] = (abs(F - Fo) / abs(Fo), grad_err(G, Go), mean_err(mu.reshape(-1), mu_o, y), np.abs(var - var_o).max() / o.prior_diag(mdo),
                       ctx.launch_count() - l0, split_err)
            mh.close()
        print(f"\nN={N}: DMMA relF {res[0][0]:.1e} relG {res[0][1]:.1e} mean {res[0][2]:.1e} var {res[0][3]:.1e} split mean {res[0][5]:.1e} | "
              f"INT8 relF {res[8][0]:.1e} relG {res[8][1]:.1e} mean {res[8][2]:.1e} var {res[8][3]:.1e} split mean {res[8][5]:.1e}")
        assert res[8][0] <= TOL_F and res[8][1] <= TOL_G and res[8][2] <= TOL_MU and res[8][3] <= TOL_VAR
        assert res[0][5] <= TOL_MU and res[8][5] <= TOL_MU
        assert res[8][4] != res[0][4]          # the route was actually taken (different launch count)
        # the inverse's W^T W on DMMA instead: fewer INT8 launches, same parity
        ctx.set_option("ozaki", 8)
        ctx.set_option("ozaki_lauum", 0)
        mh = _ffi.ModelHandle(ctx, [1, 1, 2], D, np.asfortranarray(x), y)
        l0 = ctx.launch_count()
        F, G = mh.nlml_grad(hp)
        mu, var, _ = mh.predict(xp, want_var=True)
        assert ctx.launch_count() - l0 != res[8][4]
        assert abs(F - Fo) / abs(Fo) <= TOL_F and grad_err(G, Go) <= TOL_G
        mh.close()
    finally:
        ctx.set_option("ozaki", 0)
        ctx.set_option("ozaki_lauum", 9)
        ctx.close()


# ------------------------------------------------------------------ (4) larger sizes: oracle where it is cheap, else invariants
def test_config2_n8192_three_hp_sets(gpr):
    """BASELINE.json config 2: ARD SE + noise, N=8192, D=8, FP64 NLML + gradient over 3 hp sets (SURVEY 8d).
    Oracle values are committed (tests/golden/config2_n8192.npz, make_golden_config2.py); inputs come from the seed."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mg2", os.path.join(HERE, "golden", "make_golden_config2.py"))
    mg2 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg2)
    x, y, sets = mg2.inputs()
    g = np.load(os.path.join(HERE, "golden", "config2_n8192.npz"))
    cov = gpr.SquaredExp() + gpr.WhiteNoise()
    md = gpr.GPRModel(cov, sets["A"], x, y)
    ll = gpr.MarginalLikelihood()
    tc = gpr.MllGradCache(md)
    for name, hp in sets.items():
        G = np.empty(len(hp))
        F = gpr.loss_grad_(ll, True, G, hp, md, tc)
        Fo, Go = float(g["F_" + name]), g["G_" + name]
        assert abs(F - Fo) <= TOL_F * abs(Fo), (name, F, Fo)
        assert grad_err(G, Go) <= TOL_G, (name, grad_err(G, Go))
    tc.close()


def _load_module(name, fname):
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, "golden", fname))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_config2_set_D_cond_limited(gpr):
    """SURVEY 8d config 2, set D: plain SquaredExp() (jitter only) with the hyper-parameters of set A at N = 8192.
    cond(K) ~ 1e11-1e12: the oracle value is reproduced to the cond * eps band, which is asserted as the reason."""
    mg2 = _load_module("mg2", "make_golden_config2.py")
    x, y, sets = mg2.inputs()
    g = np.load(os.path.join(HERE, "golden", "config2_n8192.npz"))
    if "F_D" not in g.files:
        pytest.skip("config2_n8192.npz predates set D")
    hp = sets["A"][:-1]
    md = gpr.GPRModel(gpr.SquaredExp(), hp, x, y)
    tc = gpr.MllGradCache(md)
    G = np.empty(len(hp))
    F = gpr.loss_grad_(gpr.MarginalLikelihood(), True, G, hp, md, tc)
    tc.close()
    cond = float(g["cond_D"])
    relF, relG = abs(F - float(g["F_D"])) / abs(float(g["F_D"])), grad_err(G, g["G_D"])
    print(f"\nconfig 2 set D: cond_est {cond:.2e}, cond*eps {cond * EPS:.1e}, relF {relF:.1e}, relG {relG:.1e}")
    assert cond * EPS > TOL_F          # the condition number IS the reason the stated 1e-8 does not apply
    assert relF <= ctol(TOL_F, cond) and relG <= ctol(TOL_G, cond)


def test_config3_n32768_benchmarked_path_vs_oracle(gpr):
    """BASELINE.json config 3 (3-ref) + config 4 at FULL size: the exact model bench.py times (N = 32768, D = 8, P = 19,
    seed 3003) through gpr_nlml_grad / gpr_fetch / gpr_predict / gpr_split_predict against oracle values committed in
    tests/golden/config3_n32768.npz (make_golden_config3.py; reference path src/cost.jl:96-127, src/predict.jl:29-95,
    src/split_predict.jl:10-53).  This is the out-of-place trtri_t + lauum_oop_t + alpha-from-inverse path."""
    path = os.path.join(HERE, "golden", "config3_n32768.npz")
    if not os.path.exists(path):
        pytest.skip("config3_n32768.npz not generated")
    mg3 = _load_module("mg3", "make_golden_config3.py")
    g = np.load(path)
    x, y, hp = mg3.inputs()
    xp, xe, xq, samp = mg3.test_inputs()
    cov = gpr.SquaredExp() + gpr.SquaredExp() + gpr.WhiteNoise()
    md = gpr.GPRModel(cov, hp, x, y)
    ll = gpr.MarginalLikelihood()
    tc = gpr.MllGradCache(md)
    G = np.empty(len(hp))
    F = gpr.loss_grad_(ll, True, G, hp, md, tc)
    Gl = np.empty(len(hp))
    Fl = gpr.log_loss_grad_(ll, True, Gl, np.log(hp), md, tc)
    alpha = tc.alpha
    tc.close()
    relF, relG, relGl = abs(F - float(g["F"])) / abs(float(g["F"])), grad_err(G, g["G"]), grad_err(Gl, g["G_log"])
    rela = np.abs(alpha - g["alpha"]).max() / np.abs(g["alpha"]).max()
    print(f"\nconfig 3 (N=32768): cond_est {float(g['cond_est']):.2e}; relF {relF:.2e}, relG {relG:.2e}, relG_log {relGl:.2e}, alpha {rela:.2e}")
    assert relF <= TOL_F and abs(Fl - float(g["F"])) <= TOL_F * abs(float(g["F"]))
    assert relG <= TOL_G and relGl <= TOL_G
    assert rela <= TOL_F
    prior = float(hp[0] ** 2 + hp[9] ** 2 + hp[18] ** 2)
    mu, Sd = gpr.predict(md, xp, diagonal_var=True)
    e_mu, e_var = mean_err(mu, g["pred_mean"], y), np.abs(Sd.diag - g["pred_var"]).max() / prior
    print(f"predict (4096 points): mean {e_mu:.2e}, var {e_var:.2e}")
    assert e_mu <= TOL_MU and e_var <= TOL_VAR
    nq = xq.shape[1]
    smu, sS = gpr.predict(md, gpr.Cmap(np.add, xe, xq), diagonal_var=True)      # default var_range = 1:3
    e_rows = mean_err(smu[:3, :], g["split_mean_rows"], y)
    e_samp = mean_err(smu.reshape(-1, order="F")[samp], g["split_mean_sampled"], y)
    e_svar = np.abs(sS.diag[:3 * nq] - g["split_var_rows"]).max() / prior
    print(f"split predict (16.8 M points): mean rows {e_rows:.2e}, sampled {e_samp:.2e}, var rows 1:3 {e_svar:.2e}")
    assert e_rows <= TOL_MU and e_samp <= TOL_MU and e_svar <= TOL_VAR
    assert np.all(sS.diag[3 * nq:3 * nq + 64] == prior)                          # rows beyond var_range keep the prior


@pytest.mark.parametrize("G", [1, 2, 4, 8])
def test_config5_n16384_distributed_vs_oracle(gpr, G):
    """SURVEY 8d config 5 parity: the block-cyclic distributed path (MultiGPUGradCache) at N = 16384, D = 16,
    SquaredExp()+WhiteNoise(), G = 1, 2, 4, 8 ranks (cycled over the visible GPUs) against the committed oracle value
    (tests/golden/config5_n16384.npz, make_golden_config5.py; reference path src/cost.jl:96-127)."""
    path = os.path.join(HERE, "golden", "config5_n16384.npz")
    if not os.path.exists(path):
        pytest.skip("config5_n16384.npz not generated")
    mg5 = _load_module("mg5", "make_golden_config5.py")
    g = np.load(path)
    x, y, hp = mg5.inputs()
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    tc = gpr.MultiGPUGradCache(md, devices=_devices(G), nb=1024)
    Gd = np.empty(len(hp))
    F = gpr.loss_grad_(gpr.MarginalLikelihood(), True, Gd, hp, md, tc)
    alpha = tc.alpha
    tc.close()
    relF, relG = abs(F - float(g["F"])) / abs(float(g["F"])), grad_err(Gd, g["G"])
    rela = np.abs(alpha - g["alpha"]).max() / np.abs(g["alpha"]).max()
    print(f"\nconfig 5 parity (N=16384, G={G}): relF {relF:.2e}, relG {relG:.2e}, alpha {rela:.2e}")
    assert relF <= TOL_F and relG <= TOL_G and rela <= TOL_F


def test_invariants_n16384(gpr):
    """Properties that need no oracle: K alpha = y, U^T U = K on sampled entries, K^-1 K = I on sampled columns,
    gradient == finite difference of the loss, determinism of repeated evaluations."""
    D, N = 8, 16384
    rng = np.random.default_rng(77)
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.5 * np.ones(D), [0.5], 2.0 * np.ones(D), [0.1]])
    cov = gpr.SquaredExp() + gpr.SquaredExp() + gpr.WhiteNoise()
    md = gpr.GPRModel(cov, hp, x, y)
    ll = gpr.MarginalLikelihood()
    tc = gpr.MllGradCache(md)
    G = np.empty(len(hp))
    F = gpr.loss_grad_(ll, True, G, hp, md, tc)
    G2 = np.empty(len(hp))
    F2 = gpr.loss_grad_(ll, True, G2, hp * (1 + 1e-15), md, tc)     # forces a re-evaluation
    assert abs(F2 - F) <= 1e-9 * abs(F)
    alpha = tc.alpha
    cols = rng.choice(N, 64, replace=False)
    Kc = o.kernel((o.SE, o.SE, o.NOISE), hp, x, x[:, cols], same=False)
    Kc[cols, np.arange(64)] += 2e-8 + hp[-1] ** 2          # jitter of both SE components + noise on the diagonal
    r = Kc.T @ alpha - y[cols]
    assert np.abs(r).max() <= 1e-9 * np.abs(y).max()
    Kinv = tc.K_inv
    E = Kinv[:, cols].T @ Kc          # rows of K^-1 times columns of K
    assert np.abs(E - np.eye(64)).max() < 1e-8
    # directional finite difference of the NLML
    v = rng.standard_normal(len(hp))
    v /= np.linalg.norm(v)
    h = 1e-5
    Fp = gpr.loss(ll, hp + h * v, md, tc)
    Fm = gpr.loss(ll, hp - h * v, md, tc)
    assert (Fp - Fm) / (2 * h) == pytest.approx(float(G @ v), rel=1e-5)
    tc.close()


# ------------------------------------------------------------------ (5) block-cyclic multi-GPU path (config 5)
# The ranks of the multi-device path cycle over the visible GPUs, so on a 1-GPU box the whole distributed code
# path (tile-mapped GEMMs, panel gathers, event barriers) runs with several ranks on cuda:0.
def _devices(G):
    from gpr_sm100a import _ffi
    nd = max(1, _ffi.device_count())
    return [r % nd for r in range(G)]


@pytest.mark.parametrize("n,nb,G", [(512, 128, 1), (768, 128, 3), (1000, 256, 2), (2048, 512, 4), (1536, 256, 8)])
def test_mgpu_dense_phases(gpr, n, nb, G):
    """potrf (+ forward solve), trtri (+ back substitution), lauum of csrc/dist_blocked.hpp against LAPACK."""
    import scipy.linalg as sl
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(n + G)
    X = rng.standard_normal((n, n))
    K = X @ X.T / n + np.eye(n)
    Y0 = rng.standard_normal((n, 3))
    U = sl.cholesky(K, lower=False)
    for mode in (0, 1, 2):
        mc = _ffi.MultiContext(_devices(G), nb=nb)
        A, Y, _ = mc.dbg_factor(np.triu(K), Y0, mode)
        mc.close()
        ref = [U, np.linalg.inv(U), np.linalg.inv(K)][mode]
        yref = sl.solve_triangular(U, Y0, trans="T") if mode == 0 else -np.linalg.solve(K, Y0)
        assert np.abs(np.triu(A) - np.triu(ref)).max() <= 1e-11 * np.abs(ref).max(), (mode,)
        assert np.abs(Y - yref).max() <= 1e-11 * np.abs(yref).max(), (mode,)
        assert not np.tril(A, -1).any()


def test_mgpu_not_positive_definite(gpr):
    from gpr_sm100a import _ffi
    K = np.eye(512)
    K[300, 300] = -2.0
    mc = _ffi.MultiContext(_devices(2), nb=128)
    with pytest.raises(gpr.PosDefException) as ei:
        mc.dbg_factor(K, None, 0)
    assert ei.value.info == 301
    mc.close()


@pytest.mark.parametrize("cov,N,D,ny,nb,G", [((o.SE, o.NOISE), 300, 5, 1, 128, 2), ((o.SE, o.SE, o.NOISE), 1000, 8, 1, 256, 3),
                                             ((o.SE, o.NOISE), 257, 3, 4, 128, 4), ((o.SE, o.MATERN52, o.NOISE), 700, 4, 1, 128, 2),
                                             ((o.SE, o.NOISE), 2000, 16, 1, 256, 8)])
def test_mgpu_nlml_grad_vs_oracle(gpr, cov, N, D, ny, nb, G):
    rng = np.random.default_rng(N + D)
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    if ny > 1:
        y = np.stack([y * (0.5 + 0.3 * k) for k in range(ny)], axis=1)
    hp = 0.3 + rng.random(o.dim_hp(cov, D))
    hp[-1] = 0.1
    ta = 2 if ny > 1 else 1
    mdo = o.GPRModel(cov, hp, x, y, train_axis=ta)
    tco = o.MllGradCache(mdo)
    Fo, Go = o.loss_grad(hp, mdo, tco)
    md = gpr.GPRModel(to_gpr_cov(gpr, cov), hp, x, y, train_axis=ta)
    tc = gpr.MultiGPUGradCache(md, devices=_devices(G), nb=nb)
    ll = gpr.MarginalLikelihood()
    Gd = np.empty(len(hp))
    F = gpr.loss_grad_(ll, True, Gd, hp, md, tc)
    assert abs(F - Fo) <= TOL_F * abs(Fo)
    assert grad_err(Gd, Go) <= TOL_G
    assert np.abs(tc.alpha - tco.alpha).max() <= 1e-8 * np.abs(tco.alpha).max()
    assert np.abs(tc.K_inv - tco.Kinv).max() <= 1e-8 * np.abs(tco.Kinv).max()
    Gl = np.empty(len(hp))
    Fl = gpr.log_loss_grad_(ll, True, Gl, np.log(hp), md, tc)
    assert abs(Fl - Fo) <= TOL_F * abs(Fo)
    assert grad_err(Gl, Go * hp) <= TOL_G
    assert gpr.loss_grad_(ll, True, None, hp, md, tc) == pytest.approx(Fo, rel=TOL_F)      # F only
    tc.close()


def test_mgpu_rank_count_independence_n8192(gpr):
    """Config 5's invariant at a size the 1-GPU box finishes quickly: F and G do not depend on the number of ranks
    or the panel width, and agree with the single-GPU path (rtol 1e-9)."""
    D, N = 16, 8192
    rng = np.random.default_rng(5005)
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.4 * np.ones(D), [0.1]])
    cov = gpr.SquaredExp() + gpr.WhiteNoise()
    md = gpr.GPRModel(cov, hp, x, y)
    ll = gpr.MarginalLikelihood()
    tc1 = gpr.MllGradCache(md)
    G1 = np.empty(len(hp))
    F1 = gpr.loss_grad_(ll, True, G1, hp, md, tc1)
    tc1.close()
    for G, nb in ((1, 1024), (2, 512), (4, 1024), (8, 256)):
        tc = gpr.MultiGPUGradCache(md, devices=_devices(G), nb=nb)
        Gd = np.empty(len(hp))
        F = gpr.loss_grad_(ll, True, Gd, hp, md, tc)
        tc.close()
        assert abs(F - F1) <= 1e-9 * abs(F1), (G, nb)
        assert grad_err(Gd, G1) <= 1e-9, (G, nb, grad_err(Gd, G1))


@pytest.mark.parametrize("G", [1, 2, 3])
def test_mgpu_int8_routes_vs_oracle(gpr, G):
    """The tile-mapped products of the block-cyclic drivers (csrc/dist_blocked.hpp) through the INT8-tensor-core product
    (csrc/ozaki_i8.cuh; nb = 1024 so that they reach the route): the rank-nb trailing updates of potrf (GEMM_MAP_UPPER) and the
    row-panel recurrence of trtri (GEMM_MAP_KUPTO: per-column contraction limit, long K cut into k-chunks with their own digit
    scales -- ozaki_kchunk = 2048 exercises the chunk loop) against the committed oracle values of config 2 (N = 8192, D = 8,
    SquaredExp()+WhiteNoise(), set A): forced on with k-chunks, automatic, forced on, potrf only, off.  The automatic rule picks
    8 digits for this model, so that leg takes the forced leg's route."""
    from gpr_sm100a import _ffi
    mg2 = _load_module("mg2", "make_golden_config2.py")
    x, y, sets = mg2.inputs()
    g = np.load(os.path.join(HERE, "golden", "config2_n8192.npz"))
    hp = sets["A"]
    launches = {}
    for forced, phases, kchunk in ((8, 11, 2048), (-1, 11, 32768), (8, 11, 32768), (8, 1, 32768), (0, 11, 32768)):
        mc = _ffi.MultiContext(_devices(G), nb=1024)
        mc.set_option("ozaki", forced)
        mc.set_option("ozaki_phases", phases)
        mc.set_option("ozaki_kchunk", kchunk)
        mm = _ffi.MultiModelHandle(mc, [1, 2], 8, x, y)
        l0 = mc.launch_count()
        F, Gd = mm.nlml_grad(hp)
        nl = mc.launch_count() - l0
        launches[(forced, phases, kchunk)] = nl
        mm.close(); mc.close()
        relF, relG = abs(F - float(g["F_A"])) / abs(float(g["F_A"])), grad_err(Gd, g["G_A"])
        print(f"\nmgpu INT8 routes, G={G}, ozaki={forced} phases={phases} kchunk={kchunk}: relF {relF:.2e} relG {relG:.2e} ({nl} launches)")
        assert relF <= TOL_F and relG <= TOL_G
    assert launches[(-1, 11, 32768)] == launches[(8, 11, 32768)]          # automatic = 8 digits: the same route
    distinct = [launches[k] for k in ((8, 11, 2048), (8, 11, 32768), (8, 1, 32768), (0, 11, 32768))]
    assert len(set(distinct)) == 4          # four different routes were actually taken


# ------------------------------------------------------------------ (6) SURVEY.md 8f "next" rows on the device
def test_update_sample_matches_oracle(gpr):
    """update_sample!(md, dy, BFGSQuad(), MarginalLikelihood(), eps_J) (src/update_model.jl:6-48, test/test_update.jl:50-76):
    same number of quasi-Newton iterations and the same re-optimised hyper-parameters as the oracle; the P + 1 gradient
    evaluations of the finite-difference Hessian spread over two caches (ReplicaGradient) give the same result."""
    import scipy.optimize as so
    rng = np.random.default_rng(11)
    D, N = 3, 120
    x = rng.random((D, N))
    hp_true = np.concatenate([[1.0], 1.0 + rng.random(D), [0.05]])
    y0 = o.sample_mvn((o.SE, o.NOISE), hp_true, x, rng.standard_normal(N))
    mdo = o.GPRModel((o.SE, o.NOISE), np.ones(D + 2), x, y0.copy())
    tco = o.MllGradCache(mdo)
    res = so.minimize(lambda v: o.log_loss_grad(v, mdo, tco), np.zeros(D + 2), jac=True, method="L-BFGS-B", options={"gtol": 1e-6, "ftol": 1e-15})
    hp_opt = np.exp(res.x)
    dy = 0.01 * y0 ** 2
    mdo.params[...] = hp_opt
    it_o = o.update_sample(mdo, dy.copy(), eps_j=1e-3)

    cov = gpr.SquaredExp() + gpr.WhiteNoise()
    ll = gpr.MarginalLikelihood()
    md = gpr.GPRModel(cov, hp_opt.copy(), x, y0.copy())
    it = gpr.update_sample_(md, dy.copy(), gpr.BFGSQuad(), ll, 1e-3)
    assert it == it_o and it < 10
    np.testing.assert_allclose(md.params, mdo.params, rtol=1e-6)
    np.testing.assert_allclose(md.y, y0 + dy)
    Gl = np.empty(D + 2)
    tc = gpr.MllGradCache(md)
    gpr.log_loss_grad_(ll, None, Gl, np.log(md.params), md, tc)
    assert np.linalg.norm(Gl) < 1e-3

    # low-level form with a second cache as a replica for the Hessian evaluations
    md2 = gpr.GPRModel(cov, hp_opt.copy(), x, y0.copy())
    tc2, rep = gpr.MllGradCache(md2), gpr.MllGradCache(md2, ctx=gpr.Context(0))
    uc = gpr.BFGSQuadCache(md2)
    it2 = gpr.update_sample_(md2, dy.copy(), ll, uc, tc2, 1e-3, replicas=[rep])
    assert it2 == it
    np.testing.assert_allclose(md2.params, md.params, rtol=1e-9)
    for c in (tc, tc2, rep):
        c.close()


@pytest.mark.parametrize("cost_name", ["MSE", "ChiSq", "Mahalanobis"])
def test_cv_batch_matches_oracle(gpr, cost_name):
    """cv_batch / cv_step! (src/crossval.jl:14-50): per fold refit + dense predictive covariance + M-estimator."""
    rng = np.random.default_rng(21)
    D, N, k = 2, 150, 10
    x = rng.random((D, N))
    y = np.sin(4 * x).sum(0) + 0.05 * rng.standard_normal(N)
    hp = np.array([1.0, 2.0, 1.5, 0.1])
    cvset = gpr.kfoldcv(N, k, 5, rng=np.random.default_rng(3))
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    lss = gpr.cv_batch(md, getattr(gpr, cost_name)(), x, y, cvset)
    cost_o = {"MSE": o.loss_mse, "ChiSq": o.loss_chisq, "Mahalanobis": o.loss_mahalanobis}[cost_name]
    lss_o = o.cv_batch(o.GPRModel((o.SE, o.NOISE), hp, x, y), cost_o, x, y, cvset)
    np.testing.assert_allclose(lss, lss_o, rtol=1e-7)
    one = gpr.cv_step(md, getattr(gpr, cost_name)(), x[:, cvset[0][2]], y[cvset[0][2]], x[:, cvset[1][2]], y[cvset[1][2]])
    assert one == pytest.approx(lss_o[2], rel=1e-7)


@pytest.mark.parametrize("cov,D,N", [((o.SE, o.NOISE), 2, 300), ((o.SE, o.SE, o.NOISE), 5, 1000), ((o.SE,), 3, 129)])
def test_sample_prior_matches_oracle(gpr, cov, D, N):
    """sample(gp(x, theta)) (src/distributions.jl:20-45) with the same normal draws: Sigma .+ 1e-7 on every entry."""
    rng = np.random.default_rng(N)
    x = rng.random((D, N))
    hp = 0.5 + rng.random(o.dim_hp(cov, D))
    z = rng.standard_normal(N)
    covo = cov if len(cov) > 1 else cov[0]
    gp = gpr.GaussianProcess(lambda col: float(np.sum(col)), to_gpr_cov(gpr, covo))
    s = gpr.sample(gp, x, hp, z=z)
    ref = o.sample_mvn(covo, hp, x, z, mu=x.sum(0))
    cond = np.linalg.cond(o.kernel(cov, hp, x) if len(cov) > 1 else o.kernel_single(cov[0], hp, x, None, True, 1e-8))
    assert np.abs(s - ref).max() <= ctol(1e-10, cond) * max(1.0, np.abs(ref).max()), (np.abs(s - ref).max(), cond)


@pytest.mark.parametrize("dim,n,ny", [(1, 100, 1), (3, 300, 4), (4, 700, 1)])
def test_integrate_matches_oracle(gpr, dim, n, ny):
    """integrate(md, hp, a, b) (src/integrate.jl:45-62,103-136, noise-free path): mean and variance of the box integral."""
    rng = np.random.default_rng(dim * 1000 + n)
    x = rng.random((dim, n))
    y = rng.random((n, ny)) if ny > 1 else rng.random(n)
    hp = np.concatenate([[1.2], 0.8 + 2.0 * rng.random(dim), [0.05]])
    a = -0.2 + 0.4 * rng.random(dim)
    b = a + 0.5 + rng.random(dim)
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    mu, var = gpr.integrate(md, hp, a, b)
    mu_o, var_o = o.integrate(o.GPRModel((o.SE, o.NOISE), hp, x, y), hp, a, b)
    np.testing.assert_allclose(mu, mu_o, rtol=1e-8, atol=1e-8 * np.abs(mu_o).max())
    assert abs(var[0] - var_o[0]) <= 1e-8 * o.antideriv2(hp, a, b)
    # per-sample-noise branch (src/integrate.jl:72-100,145-160): the oracle follows the reference's eigendecomposition,
    # the device takes one shifted Cholesky per noise level -- same quantities
    noise = 1e-3 * (1.0 + rng.random(max(ny, 1)))
    mu_n, var_n = gpr.integrate(md, hp, a, b, sample_noise=noise)
    mu_no, var_no = o.integrate(o.GPRModel((o.SE, o.NOISE), hp, x, y), hp, a, b, noise)
    np.testing.assert_allclose(mu_n, mu_no, rtol=1e-7, atol=1e-8 * np.abs(mu_no).max())
    np.testing.assert_allclose(var_n, var_no, rtol=0, atol=1e-7 * o.antideriv2(hp, a, b))
    mu_s, var_s = gpr.integrate(md, hp, a, b, sample_noise=2e-3)
    mu_so, var_so = o.integrate(o.GPRModel((o.SE, o.NOISE), hp, x, y), hp, a, b, 2e-3)
    np.testing.assert_allclose(mu_s, mu_so, rtol=1e-7, atol=1e-8 * np.abs(mu_so).max())
    np.testing.assert_allclose(var_s, np.broadcast_to(var_so, var_s.shape), rtol=0, atol=1e-7 * o.antideriv2(hp, a, b))


def test_integrate_agrees_with_quadrature_of_the_posterior_mean(gpr):
    """Property (no oracle): the analytic integral of the posterior mean equals Gauss-Legendre quadrature of
    predict_mean over the box (cf. test/test_integrate.jl:164-177)."""
    rng = np.random.default_rng(6)
    dim, n = 2, 400
    x = rng.random((dim, n))
    y = np.sin(x.prod(0)) ** 2
    hp = np.array([1.0, 1.5, 1.5, 0.01])
    md = gpr.GPRModel(gpr.SquaredExp() + gpr.WhiteNoise(), hp, x, y)
    mu, var = gpr.integrate(md, np.zeros(dim), np.ones(dim))
    xg, wg = np.polynomial.legendre.leggauss(24)
    xg, wg = 0.5 * (xg + 1), 0.5 * wg
    grid = np.asfortranarray(np.stack(np.meshgrid(xg, xg, indexing="ij")).reshape(2, -1))
    W = np.outer(wg, wg).ravel()
    pm = gpr.predict_mean(md, grid)
    assert mu[0] == pytest.approx(float(W @ pm), rel=1e-9)
    assert var[0] >= -1e-10


# ------------------------------------------------------------------ (7) edge sizes
@pytest.mark.parametrize("N", [1, 2, 3, 127, 128, 129])
def test_tiny_and_boundary_sizes(gpr, N):
    """Sizes around the 128-padding boundary and degenerate training sets (the reference has no lower limit on n)."""
    rng = np.random.default_rng(N)
    D = 2
    x = rng.random((D, N))
    y = rng.random(N)
    hp = np.array([1.1, 0.9, 1.3, 0.2])
    cov, covo = gpr.SquaredExp() + gpr.WhiteNoise(), (o.SE, o.NOISE)
    md, mdo = gpr.GPRModel(cov, hp, x, y), o.GPRModel(covo, hp, x, y)
    ll = gpr.MarginalLikelihood()
    tc = gpr.MllGradCache(md)
    G = np.empty(4)
    F = gpr.loss_grad_(ll, True, G, hp, md, tc)
    Fo, Go = o.loss_grad(hp, mdo)
    assert abs(F - Fo) <= TOL_F * max(abs(Fo), 1.0)
    assert np.abs(G - Go).max() <= TOL_G * max(np.abs(Go).max(), 1.0)
    tc.close()
    xp = rng.random((D, 5))
    mu, Sig = gpr.predict(md, xp, diagonal_var=True)
    mu_o, var_o = o.predict(mdo, xp, diagonal_var=True)
    assert np.abs(mu - mu_o).max() <= TOL_MU * max(np.abs(mu_o).max(), 1.0)
    assert np.abs(Sig.diag - var_o).max() <= TOL_VAR * o.prior_diag(mdo)
    tcm = gpr.MultiGPUGradCache(md, devices=_devices(2), nb=128)
    Gm = np.empty(4)
    Fm = gpr.loss_grad_(ll, True, Gm, hp, md, tcm)
    assert abs(Fm - Fo) <= TOL_F * max(abs(Fo), 1.0)
    assert np.abs(Gm - Go).max() <= TOL_G * max(np.abs(Go).max(), 1.0)
    tcm.close()


def test_mgpu_prefetch_modes_agree(gpr):
    """The three transports of the prefetched panels (main queue / SM pulls / copy engines) give identical results."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(9)
    n = 1536
    X = rng.standard_normal((n, n))
    K = X @ X.T / n + np.eye(n)
    Y0 = rng.standard_normal((n, 2))
    outs = []
    for mode in (0, 1, 2):
        mc = _ffi.MultiContext(_devices(3), nb=256)
        mc.set_option("prefetch_trtri", mode)
        mc.set_option("prefetch_lauum", mode)
        A, Y, _ = mc.dbg_factor(np.triu(K), Y0, 2)
        mc.close()
        outs.append((A, Y))
    for A, Y in outs[1:]:
        assert np.array_equal(A, outs[0][0]) and np.array_equal(Y, outs[0][1])
    assert np.abs(np.triu(outs[0][0]) - np.triu(np.linalg.inv(K))).max() <= 1e-11 * np.abs(np.linalg.inv(K)).max()


def test_mgpu_packed_transport_matches_peer_transport(gpr):
    """Transport 1 runs the pack -> collective -> unpack data path of the NCCL transport (gpr_dist_create) with in-process
    copies as the collective: same arithmetic, so the results must equal the peer-memory transport bit for bit."""
    from gpr_sm100a import _ffi
    rng = np.random.default_rng(31)
    n = 1280
    X = rng.standard_normal((n, n))
    K = X @ X.T / n + np.eye(n)
    Y0 = rng.standard_normal((n, 2))
    res = []
    for transport in (0, 1):
        mc = _ffi.MultiContext(_devices(3), nb=256, transport=transport)
        A, Y, _ = mc.dbg_factor(np.triu(K), Y0, 2)
        mc.close()
        res.append((A, Y))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    # model level: F, G, alpha through the packed transport vs the oracle
    D, N = 4, 900
    x = rng.random((D, N))
    y = np.sin(3 * x).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], 0.6 * np.ones(D), [0.1]])
    Fo, Go = o.loss_grad(hp, o.GPRModel((o.SE, o.NOISE), hp, x, y))
    mc = _ffi.MultiContext(_devices(4), nb=128, transport=1)
    mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
    F, G = mm.nlml_grad(hp)
    Fl, _ = mm.nlml_grad(hp, want_g=False)
    assert abs(F - Fo) <= TOL_F * abs(Fo) and abs(Fl - Fo) <= TOL_F * abs(Fo)
    assert grad_err(G, Go) <= TOL_G
    mm.close(); mc.close()
