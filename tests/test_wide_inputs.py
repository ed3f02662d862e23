"""High-dimensional inputs: the chunked covariance build (kbuild_kernel<MODE, true>) and the wide gradient reduction
(csrc/grad_wide.cuh) take every shape whose point tiles or per-thread accumulators do not fit in shared memory.

Length scales are l_d ~ U(0.5, 1.5) / sqrt(D) (inverse length scales, as the library reads them) so that distances are
O(1) at every D: otherwise K is nearly diagonal and the gradient checks say nothing.  Tolerances are those of
tests/test_gpu_parity.py (TOL 1e-8, raised to 10 cond(K) eps where that is larger)."""
import os

import numpy as np
import pytest

import gpr_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
EPS = 2.2e-16
TOL_F, TOL_G, TOL_MU, TOL_VAR = 1e-8, 1e-8, 1e-8, 1e-8
TYPES = {o.SE: 1, o.NOISE: 2, o.MATERN52: 3}


def ctol(stated, cond):
    return max(stated, 10.0 * cond * EPS)


def grad_err(G, Gref):
    return float((np.abs(G - Gref) / np.maximum(np.abs(Gref), 1e-8 * np.linalg.norm(Gref))).max())


def mean_err(mu, ref, y):
    return float((np.abs(mu - ref) / np.maximum(np.abs(ref), 1e-8 * np.abs(y).max())).max())


def wide_problem(cov, N, D, seed, ny=1):
    rng = np.random.default_rng(seed)
    x = np.asfortranarray(rng.random((D, N)))
    y = np.sin(3 * x[: min(D, 16)]).sum(0) + 0.1 * rng.standard_normal(N)
    if ny > 1:
        y = np.asfortranarray(np.stack([y * (0.5 + 0.3 * k) for k in range(ny)], axis=1))
    hp = []
    for c in cov:
        if c == o.NOISE:
            hp.append([0.3])
        else:
            hp.append(np.concatenate([[0.5 + rng.random()], rng.uniform(0.5, 1.5, D) / np.sqrt(D)]))
    return x, y, np.concatenate(hp), rng


def takes_wide_build(cov, D):
    """launch_kbuild takes kbuild_kernel<MODE, true> (the point tiles of all components exceed 200 KB of shared memory)"""
    nk = sum(1 for c in cov if c != o.NOISE)
    return 2 * nk * D * 64 * 8 > 200 * 1024


def takes_wide_grad(cov, D):
    """launch_grad_reduce takes grad_reduce_wide_kernel (per-thread accumulators and point tiles exceed 200 KB)"""
    P = o.dim_hp(cov, D)
    return ((P + 1) * 256 + 128 * D + 160) * 8 > 200 * 1024


def pair_sums(M, xr, xc):
    """s_d = sum_ab M_ab (xr_da - xc_db)^2 through the translation-invariant identity on coordinates centred on xr[:, 0]:
    sum_a u_ad^2 R_a + sum_b v_bd^2 C_b - 2 sum_a u_ad (M V)_ad (csrc/grad_wide.cuh)"""
    c = xr[:, :1]
    u, v = (xr - c).T, (xc - c).T
    R, Cs = M.sum(1), M.sum(0)
    return (u * u).T @ R + (v * v).T @ Cs - 2.0 * np.einsum("ad,ad->d", u, M @ v)


def direct_pair_sums(M, x):
    """s_d = sum_ab M_ab (x_ad - x_bd)^2 term by term (independent of the identity the wide gradient uses)"""
    return np.array([(M * (x[d][:, None] - x[d][None, :]) ** 2).sum() for d in range(x.shape[0])])


def ref_loss_grad(cov, hp, x, y, train_axis=1, eps=1e-8, direct=False):
    """F and G of the oracle (loss_grad.jl:40-52), the length-scale terms summed by pair_sums over the full matrix, or term
    by term with direct=True"""
    import scipy.linalg as sl
    D = x.shape[0]
    K = o.kernel(cov, hp, x)
    U = sl.cholesky(K, lower=False)
    yy = y.reshape(y.shape[0], -1)
    alpha = sl.cho_solve((U, False), yy)[:, train_axis - 1]
    yt = yy[:, train_axis - 1]
    F = 0.5 * (yt @ alpha + 2 * np.log(np.diag(U)).sum() + len(yt) * np.log(2 * np.pi))
    Kinv = sl.cho_solve((U, False), np.eye(len(yt)))
    W = np.outer(alpha, alpha) - Kinv
    G = np.zeros(len(hp))
    off = 0
    for c in cov:
        if c == o.NOISE:
            G[off] = -hp[off] * np.trace(W)
            off += 1
            continue
        sg, ls = hp[off], hp[off + 1:off + 1 + D]
        xs = x * ls[:, None]
        sq = (xs * xs).sum(0)
        d2 = np.maximum(sq[:, None] + sq[None, :] - 2 * xs.T @ xs, 0.0)
        np.fill_diagonal(d2, 0.0)
        if c == o.SE:
            Kc = sg * sg * np.exp(-d2) + eps * np.eye(len(yt))
            KL = Kc
        else:
            r5 = np.sqrt(5.0 * d2)
            e = np.exp(-r5)
            Kc = sg * sg * (1 + r5 + 5.0 / 3.0 * d2) * e + eps * np.eye(len(yt))
            KL = 5.0 / 6.0 * sg * sg * (1 + r5) * e
        G[off] = -(W * Kc).sum() / abs(sg)
        G[off + 1:off + 1 + D] = ls * (direct_pair_sums(W * KL, x) if direct else pair_sums(W * KL, x, x))
        off += 1 + D
    return F, G, np.linalg.cond(K)


# ----------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("shift", [0.0, 1000.0])
def test_tile_contraction_identity(shift):
    """The per-tile contraction of the wide gradient against the direct sum_ab M_ab (x_ad - x_bd)^2: a diagonal tile with
    upper-only storage (diagonal weight 1, 2 above, 0 below), an off-diagonal tile, padded rows, shifted inputs."""
    rng = np.random.default_rng(5)
    D = 37
    x = shift + rng.random((D, 128))
    x0 = x[:, :1]
    for (ti, tj) in ((0, 0), (0, 1), (1, 1)):
        xr, xc = x[:, 64 * ti:64 * ti + 64], x[:, 64 * tj:64 * tj + 64]
        M = rng.standard_normal((64, 64))
        if ti == tj:
            M = np.triu(M) + np.triu(M, 1)           # weight 2 above the diagonal, 1 on it, 0 below
        M[50:, :] = 0.0                              # rows beyond N
        direct = np.einsum("ab,dab->d", M, (xr[:, :, None] - xc[:, None, :]) ** 2)
        c = x0
        u, v = (xr - c).T, (xc - c).T
        ident = (u * u).T @ M.sum(1) + (v * v).T @ M.sum(0) - 2.0 * np.einsum("ad,ad->d", u, M @ v)
        scale = np.einsum("ab,dab->d", np.abs(M), (xr[:, :, None] - xc[:, None, :]) ** 2)
        assert np.all(np.abs(ident - direct) <= 1e-13 * scale), (ti, tj, np.abs(ident - direct).max())


def test_tile_contraction_needs_the_centre():
    """Without the centre the three terms are each of the size of |x|^2 and cancel: at x + 1000 the uncentred form loses
    digits the centred one keeps."""
    rng = np.random.default_rng(6)
    D = 16
    xr, xc = 1000.0 + rng.random((D, 64)), 1000.0 + rng.random((D, 64))
    M = rng.standard_normal((64, 64))
    direct = np.einsum("ab,dab->d", M, (xr[:, :, None] - xc[:, None, :]) ** 2)
    u, v = xr.T, xc.T
    raw = (u * u).T @ M.sum(1) + (v * v).T @ M.sum(0) - 2.0 * np.einsum("ad,ad->d", u, M @ v)
    cen = pair_sums(M, xr, xc)
    assert np.abs(cen - direct).max() <= 1e-12 * np.abs(direct).max()
    assert np.abs(raw - direct).max() > 1e-9 * np.abs(direct).max()


@pytest.mark.parametrize("cov", [(o.SE, o.SE, o.NOISE), (o.SE, o.MATERN52, o.NOISE)])
def test_reference_gradient_matches_oracle(cov):
    """ref_loss_grad (used below at sizes where the oracle's dense dK loop is slow) is the oracle's F and G"""
    x, y, hp, _ = wide_problem(cov, 150, 12, 3)
    F, G, _ = ref_loss_grad(cov, hp, x, y)
    Fd, Gd, _ = ref_loss_grad(cov, hp, x, y, direct=True)
    Fo, Go = o.loss_grad(hp, o.GPRModel(cov, hp, x, y))
    assert F == pytest.approx(Fo, rel=1e-12) and Fd == F
    assert grad_err(G, Go) <= 1e-10 and grad_err(Gd, Go) <= 1e-10


# ----------------------------------------------------------------------------------------------------------- GPU
def _ctx(**options):
    from gpr_sm100a import _ffi
    ctx = _ffi.Context(0)
    for k, v in options.items():
        ctx.set_option(k, v)
    return ctx


@pytest.mark.gpu
def test_zero_padding_is_invisible(gpr):
    """SE + noise at D = 8 (shared-memory kernels) against the same points padded with 248 zero coordinates (chunked build,
    wide gradient): the same F, G and predictions; the gradient of every padded length scale is exactly 0."""
    from gpr_sm100a import _ffi
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = wide_problem(cov, 1000, 8, 11)
    D2 = 256
    assert takes_wide_build(cov, D2) and takes_wide_grad(cov, D2) and not takes_wide_build(cov, 8)
    xpad = np.asfortranarray(np.concatenate([x, np.zeros((D2 - 8, x.shape[1]))]))
    hp_pad = np.concatenate([hp[:9], rng.uniform(0.5, 1.5, D2 - 8), hp[9:]])
    xp = np.asfortranarray(rng.random((8, 400)))
    xpp = np.asfortranarray(np.concatenate([xp, np.zeros((D2 - 8, 400))]))
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    ctx = _ctx()
    try:
        m1 = _ffi.ModelHandle(ctx, [1, 2], 8, x, y)
        m2 = _ffi.ModelHandle(ctx, [1, 2], D2, xpad, y)
        F1, G1 = m1.nlml_grad(hp)
        F2, G2 = m2.nlml_grad(hp_pad)
        assert F2 == pytest.approx(F1, rel=ctol(TOL_F, cond))
        G2s = np.concatenate([G2[:9], G2[-1:]])
        assert grad_err(G2s, G1) <= ctol(TOL_G, cond)
        assert np.all(G2[9:-1] == 0.0)
        mu1, v1, _ = m1.predict(xp, want_var=True)
        mu2, v2, _ = m2.predict(xpp, want_var=True)
        assert mean_err(mu2.ravel(), mu1.ravel(), y) <= ctol(TOL_MU, cond)
        assert np.abs(v2 - v1).max() <= ctol(TOL_VAR, cond) * (hp[0] ** 2 + hp[-1] ** 2)
    finally:
        ctx.close()


# (composition, N, D, ny, train_axis)
PARITY = [((o.SE, o.NOISE), 1000, 65, 1, 1), ((o.SE, o.NOISE), 2048, 96, 1, 1), ((o.SE, o.NOISE), 1000, 300, 1, 1),
          ((o.SE, o.NOISE), 2048, 300, 1, 1), ((o.SE, o.SE, o.NOISE), 1000, 40, 1, 1),
          ((o.SE, o.MATERN52, o.NOISE), 1000, 128, 1, 1), ((o.SE, o.NOISE), 1024, 1024, 1, 1), ((o.SE, o.NOISE), 1000, 128, 3, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("cov,N,D,ny,ta", PARITY)
def test_wide_loss_grad_parity(gpr, cov, N, D, ny, ta):
    from gpr_sm100a import _ffi
    x, y, hp, _ = wide_problem(cov, N, D, N + D + ny, ny)
    # D = 300: the length-scale terms of the reference summed term by term, not through the identity under test
    Fo, Go, cond = ref_loss_grad(cov, hp, x, y, ta, direct=(N, D) == (1000, 300))
    assert takes_wide_grad(cov, D)
    ctx = _ctx()
    try:
        m = _ffi.ModelHandle(ctx, [TYPES[c] for c in cov], D, x, y, ta)
        F, G = m.nlml_grad(hp)
        print(f"\n{cov} N={N} D={D}: relF {abs(F - Fo) / abs(Fo):.1e} relG {grad_err(G, Go):.1e} cond {cond:.1e}")
        assert F == pytest.approx(Fo, rel=ctol(TOL_F, cond))
        assert grad_err(G, Go) <= ctol(TOL_G, cond)
        for i in (0, 1, D // 2, len(hp) - 1):           # finite differences (test_loss_reference_suite)
            hpe = hp.copy()
            hpe[i] += 1e-6
            Fe, _ = m.nlml_grad(hpe, want_g=False)
            fd = (Fe - F) / 1e-6
            assert G[i] == pytest.approx(fd, rel=2e-3, abs=1e-3 * max(1.0, abs(fd)))
        if (N, D) == (1000, 300):                      # determinism: the same bits twice
            F2, G2 = m.nlml_grad(hp)
            assert F2 == F and np.array_equal(G2, G)
        m.close()
    finally:
        ctx.close()


@pytest.mark.gpu
def test_wide_shifted_inputs(gpr):
    """x + 1000 at D = 128: the centred contractions keep the digits (without centring about 12 of them are lost)"""
    from gpr_sm100a import _ffi
    cov = (o.SE, o.NOISE)
    x, y, hp, _ = wide_problem(cov, 1000, 128, 21)
    xs = np.asfortranarray(x + 1000.0)
    Fo, Go, cond = ref_loss_grad(cov, hp, x, y)                  # distances do not depend on the shift
    ctx = _ctx()
    try:
        m = _ffi.ModelHandle(ctx, [1, 2], 128, xs, y)
        F, G = m.nlml_grad(hp)
        print(f"\nshifted: relF {abs(F - Fo) / abs(Fo):.1e} relG {grad_err(G, Go):.1e}")
        # the build takes direct differences of the shifted coordinates (1e3 * eps of rounding per coordinate)
        assert F == pytest.approx(Fo, rel=ctol(1e-7, cond))
        assert grad_err(G, Go) <= ctol(1e-7, cond)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cov,D", [((o.SE, o.NOISE), 256), ((o.SE, o.MATERN52, o.NOISE), 128)])
def test_wide_entry_points(gpr, cov, D):
    """Every builder on the chunked covariance build: predict (mean with the fused K* mean, Diagonal, dense), the strict lower
    triangle of the cached factor (lower_only), gpr_kernel, prior sampling (all_shift), and for SquaredExp models split
    predict (split A / B / C factors).  Box integration: test_wide_integrate."""
    from gpr_sm100a import _ffi
    import scipy.linalg as sl
    assert takes_wide_build(cov, D)
    types = [TYPES[c] for c in cov]
    x, y, hp, rng = wide_problem(cov, 1000, D, 31)
    mdo = o.GPRModel(cov, hp, x, y)
    Ko = o.kernel(cov, hp, x)
    cond = np.linalg.cond(Ko)
    ctx = _ctx()
    try:
        m = _ffi.ModelHandle(ctx, types, D, x, y)
        m.update_cache(hp)
        xp = np.asfortranarray(rng.random((D, 300)))
        mu_o, Sig_o = o.predict(mdo, xp)
        _, var_o = o.predict(mdo, xp, diagonal_var=True)
        mu_m, _, _ = m.predict(xp)                       # mean only: K* is not stored, its mean fused into the build
        mu, var, Sig = m.predict(xp, want_var=True, want_cov=True)
        pd = o.prior_diag(mdo)
        assert mean_err(mu_m.ravel(), mu_o, y) <= ctol(TOL_MU, cond)
        assert mean_err(mu.ravel(), mu_o, y) <= ctol(TOL_MU, cond)
        assert np.abs(var - var_o).max() <= ctol(TOL_VAR, cond) * pd
        assert np.abs(Sig - Sig_o).max() <= ctol(TOL_VAR, cond) * pd
        U = m.fetch(_ffi.FETCH_U)                         # strict lower triangle: K, filled in on demand
        assert np.abs(np.tril(U, -1) - np.tril(Ko, -1)).max() <= 1e-12 * np.abs(Ko).max()
        if o.MATERN52 not in cov:
            xe, xq = np.asfortranarray(0.5 * rng.random((D, 12))), np.asfortranarray(0.5 * rng.random((D, 9)))
            smu_o, svar_o = o.split_predict(mdo, o.Cmap(xe, xq), var_range=(1, 12))
            smu, svar = m.split_predict(xe, xq, var_range=(1, 12))
            assert mean_err(smu.ravel(), smu_o.ravel(), y) <= ctol(TOL_MU, cond)
            assert np.abs(svar.ravel() - svar_o).max() <= ctol(TOL_VAR, cond) * pd
        m.close()
        K = _ffi.kernel_matrix(ctx, types, D, hp, x, xp, False, 1e-8, False)
        Kxo = o.kernel(cov, hp, x, xp)
        assert np.abs(K - Kxo).max() <= 1e-12 * np.abs(Kxo).max()
        xs = np.asfortranarray(x[:, :300])
        z = rng.standard_normal(300)
        s = _ffi.sample_mvn(ctx, types, D, hp, xs, z)
        so = o.sample_mvn(cov, hp, xs, z)
        assert np.abs(s - so).max() <= 1e-8 * np.abs(so).max()
    finally:
        ctx.close()


def box_problem(N, D, seed):
    """SE + noise with inverse length scales U(0.5, 1.5) on points in a cube of side 1.6 / sqrt(D) (distances O(1)) and 10
    boxes of width about 1 around them.  antideriv! (integrate.jl:15-31) carries prod (sqrt(pi)/2)/l_i and
    the product of the erf differences apart, so each stays within the double range only for length scales like these:
    with l ~ 1/sqrt(D) the first overflows beyond D of a few hundred, in the reference's arithmetic as in this library's."""
    rng = np.random.default_rng(seed)
    side = 1.6 / np.sqrt(D)
    x = np.asfortranarray(0.5 + side * (rng.random((D, N)) - 0.5))
    y = np.sin(3 * x[:16] / side).sum(0) + 0.1 * rng.standard_normal(N)
    hp = np.concatenate([[1.0], rng.uniform(0.5, 1.5, D), [0.3]])
    w = 1.0 + 0.05 * rng.standard_normal((D, 10))
    c = 0.5 + 0.05 * rng.standard_normal((D, 10))
    return x, y, hp, np.asfortranarray(c - 0.5 * w), np.asfortranarray(c + 0.5 * w)


def check_boxes(I, ivar, x, y, hp, cov, a, b, cond):
    """Iout and variance of every box against the oracle's antideriv / antideriv2 and a LAPACK factor (src/integrate.jl)"""
    import scipy.linalg as sl
    U = sl.cholesky(o.kernel(cov, hp, x), lower=False)
    wt = sl.cho_solve((U, False), y)
    for i in range(a.shape[1]):
        k1 = o.antideriv(x, hp, a[:, i], b[:, i])
        k2 = o.antideriv2(hp, a[:, i], b[:, i])
        assert np.isfinite(k2) and k2 > 0
        tt = sl.solve_triangular(U, k1, trans="T", lower=False)
        assert I[i, 0] == pytest.approx(wt @ k1, rel=ctol(1e-8, cond))
        assert abs(ivar[i] - (k2 - tt @ tt)) <= ctol(1e-8, cond) * k2


@pytest.mark.gpu
@pytest.mark.parametrize("D,N", [(256, 1000), (1024, 1000), (2048, 256)])
def test_wide_integrate(gpr, D, N):
    """gpr_integrate_batch and gpr_integrate at D = 256 and 1024 (the bounds of 8 boxes, up to 128 KB, in shared memory at
    once) and D = 2048 (256 KB: over the 227 KB a CTA can have, staged in chunks of coordinates); gpr_mgpu_integrate on two
    ranks at D = 2048"""
    from gpr_sm100a import _ffi
    cov = (o.SE, o.NOISE)
    x, y, hp, a, b = box_problem(N, D, 71 + D)
    cond = np.linalg.cond(o.kernel(cov, hp, x))
    ctx = _ctx()
    try:
        m = _ffi.ModelHandle(ctx, [1, 2], D, x, y)
        m.update_cache(hp)
        I, ivar = m.integrate(a, b)
        check_boxes(I, ivar, x, y, hp, cov, a, b, cond)
        I1, v1 = m.integrate(np.ascontiguousarray(a[:, 3]), np.ascontiguousarray(b[:, 3]))
        check_boxes(I1.reshape(1, -1), v1, x, y, hp, cov, a[:, 3:4], b[:, 3:4], cond)
        m.close()
    finally:
        ctx.close()
    if D == 2048:
        mc = _ffi.MultiContext([0, 0], nb=128)
        try:
            mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
            mm.update_cache(hp)
            Im, vm = mm.integrate(a, b)
            check_boxes(Im, vm, x, y, hp, cov, a, b, cond)
            mm.close()
        finally:
            mc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("G,transport", [(1, 0), (2, 0), (2, 1)])
def test_wide_mgpu(gpr, G, transport):
    """gpr_mgpu_nlml_grad and gpr_mgpu_predict at D = 256 (the listed device taken G times; chunked row-block build, wide
    gradient) against the single-GPU model and the oracle"""
    from gpr_sm100a import _ffi
    cov, D = (o.SE, o.NOISE), 256
    assert takes_wide_build(cov, D) and takes_wide_grad(cov, D)
    x, y, hp, rng = wide_problem(cov, 1000, D, 41)
    Fo, Go, cond = ref_loss_grad(cov, hp, x, y)
    xp = np.asfortranarray(rng.random((D, 200)))
    mu_o, var_o = o.predict(o.GPRModel(cov, hp, x, y), xp, diagonal_var=True)
    ctx = _ctx()
    try:
        m = _ffi.ModelHandle(ctx, [1, 2], D, x, y)
        F1, G1 = m.nlml_grad(hp)
        m.close()
    finally:
        ctx.close()
    mc = _ffi.MultiContext([0] * G, nb=256, transport=transport)
    try:
        mm = _ffi.MultiModelHandle(mc, [1, 2], D, x, y)
        F, Gm = mm.nlml_grad(hp)
        assert F == pytest.approx(Fo, rel=ctol(TOL_F, cond)) and F == pytest.approx(F1, rel=ctol(TOL_F, cond))
        assert grad_err(Gm, Go) <= ctol(TOL_G, cond) and grad_err(Gm, G1) <= ctol(TOL_G, cond)
        mu, var, _ = mm.predict(xp, want_var=True)
        assert mean_err(mu.ravel(), mu_o, y) <= ctol(TOL_MU, cond)
        assert np.abs(var - var_o).max() <= ctol(TOL_VAR, cond) * (hp[0] ** 2 + hp[-1] ** 2)
        mm.close()
    finally:
        mc.close()


@pytest.mark.gpu
def test_wide_int8_route(gpr):
    """N = 8192, D = 128: the INT8 product route (ozaki forced) against DMMA products, within the route's tolerances"""
    from gpr_sm100a import _ffi
    cov, D, N = (o.SE, o.NOISE), 128, 8192
    x, y, hp, _ = wide_problem(cov, N, D, 51)
    res = {}
    for oz in (0, 8):
        ctx = _ctx(ozaki=oz, ozaki_min=512)
        try:
            m = _ffi.ModelHandle(ctx, [1, 2], D, x, y)
            l0 = ctx.launch_count()
            res[oz] = m.nlml_grad(hp) + (ctx.launch_count() - l0,)
            m.close()
        finally:
            ctx.close()
    (F0, G0, l0), (F8, G8, l8) = res[0], res[8]
    print(f"\nINT8 vs DMMA at D={D}: relF {abs(F8 - F0) / abs(F0):.1e} relG {grad_err(G8, G0):.1e}")
    assert l8 != l0
    assert abs(F8 - F0) <= TOL_F * abs(F0)
    assert grad_err(G8, G0) <= TOL_G


@pytest.mark.gpu
def test_narrow_shapes_unchanged(gpr):
    """Shapes that the shared-memory kernels take run the same kernels with the same bits and the same launch count as the
    library before the wide-input kernels (tests/golden/parent/narrow_calls.npz, make_golden_narrow.py)"""
    import importlib.util
    from gpr_sm100a import _ffi
    spec = importlib.util.spec_from_file_location("mgn", os.path.join(HERE, "golden", "make_golden_narrow.py"))
    mgn = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mgn)
    ref = np.load(os.path.join(HERE, "golden", "parent", "narrow_calls.npz"))
    got = mgn.calls(_ffi)
    assert sorted(got) == sorted(ref.files)
    for k in ref.files:
        assert np.array_equal(got[k], ref[k]), k


@pytest.mark.gpu
def test_creation_takes_every_width(gpr):
    """D = 1024 with seven SquaredExp components and noise (P = 7176, eight components) is created, factored and differentiated"""
    from gpr_sm100a import _ffi
    D, N = 1024, 256
    cov = (o.SE,) * 7 + (o.NOISE,)
    x, y, hp, _ = wide_problem(cov, N, D, 61)
    ctx = _ctx()
    try:
        m = _ffi.ModelHandle(ctx, [TYPES[c] for c in cov], D, x, y)
        F, G = m.nlml_grad(hp)
        Fo, Go, cond = ref_loss_grad(cov, hp, x, y)
        assert len(G) == 7 * (D + 1) + 1
        assert F == pytest.approx(Fo, rel=ctol(TOL_F, cond))
        assert grad_err(G, Go) <= ctol(TOL_G, cond)
        m.close()
    finally:
        ctx.close()
