"""Split prediction on Cmap(+, xe, xq) grids on the block-cyclic multi-GPU model (gpr_mgpu_split_predict, pytest -m gpu).
The ranks cycle over the visible GPUs, so a 1-GPU box runs the whole distributed path with several ranks on cuda:0.
Tolerances as in tests/test_mgpu_predict.py."""
import os

import numpy as np
import pytest

import gpr_oracle as o
from test_mgpu_predict import TOL_MU, TOL_VAR, _cond_bound, _devices, ctol, mean_err, problem, to_gpr_cov

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def grid(rng, D, ne, nq):
    return 0.5 * rng.random((D, ne)), 0.5 * rng.random((D, nq))


def cond_of(cov, hp, x):
    return np.linalg.cond(o.kernel(cov, hp, x))


def mgpu_model(x, y, types, G, nb, transport=0, ozaki=None, tile=None):
    from gpr_sm100a import _ffi
    mc = _ffi.MultiContext(_devices(G), nb=nb, transport=transport)
    if ozaki is not None:
        mc.set_option("ozaki", ozaki)
    if tile is not None:
        mc.set_option("predict_tile", tile)
    return mc, _ffi.MultiModelHandle(mc, types, x.shape[0], x, y)


TYPES = {o.SE: 1, o.NOISE: 2, o.MATERN52: 3}

# (composition, N, D, nb, G): N = 300 with nb = 128 on 8 ranks leaves ranks without a block; N is no multiple of nb
CASES = [((o.SE, o.NOISE), 300, 3, 128, 8), ((o.SE, o.NOISE), 1000, 4, 256, 2), ((o.SE, o.SE, o.NOISE), 700, 2, 128, 3),
         ((o.SE, o.SE), 400, 3, 256, 1), ((o.SE, o.SE, o.NOISE), 500, 5, 256, 2)]


@pytest.mark.parametrize("cov,N,D,nb,G", CASES)
def test_mgpu_split_vs_oracle(gpr, cov, N, D, nb, G):
    x, y, hp, rng = problem(cov, N, D, 1, N + 3 * G + nb)
    mdo = o.GPRModel(cov, hp, x, y)
    cond = cond_of(cov, hp, x)
    prior = o.prior_diag(mdo)
    mc, mm = mgpu_model(x, y, [TYPES[c] for c in cov], G, nb)
    mm.update_cache(hp)
    xe, xq = grid(rng, D, 37, 300)   # ne, nq no multiples of 128; nq < 128 G at G = 3, 8
    mean_only, _ = mm.split_predict(xe, xq, want_var=False)
    for vr in ((1, 3), (5, 9), (1, 0)):
        mu, var = mm.split_predict(xe, xq, var_range=vr)
        mu_o, var_o = o.split_predict(mdo, o.Cmap(xe, xq), var_range=vr)
        assert np.array_equal(mu, mean_only)            # the variance rows do not touch the mean
        assert mean_err(mu, mu_o, y) <= ctol(TOL_MU, cond)
        assert np.abs(var - var_o).max() <= ctol(TOL_VAR, cond) * prior
        rows = np.zeros(37, bool)
        rows[vr[0] - 1:vr[1]] = True
        assert np.all(var.reshape(37, 300)[~rows] == prior)
    mm.close(); mc.close()


def _single_split(gpr, x, y, hp, types, xe, xq, ozaki, var_range=None):
    from gpr_sm100a import _ffi
    ctx = _ffi.Context(0)
    ctx.set_option("ozaki", ozaki)
    mh = _ffi.ModelHandle(ctx, types, x.shape[0], x, y)
    mh.update_cache(hp)
    out = mh.split_predict(xe, xq, var_range=var_range, want_var=var_range is not None)
    mh.close(); ctx.close()
    return out


def test_mgpu_split_mean_bit_identical_across_ranks_transports_chunks(gpr):
    """DMMA products ("ozaki" = 0): every output element of the mean takes the same k order whatever the column partition,
    so the mean does not depend on the number of ranks, the transport or the slab width (predict_tile 128: several chunks)."""
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 1500, 4, 1, 41)
    xe, xq = grid(rng, 4, 200, 1100)
    ref = None
    for G, transport, tile in ((1, 0, None), (2, 0, None), (4, 0, None), (2, 1, None), (4, 1, 128), (3, 0, 128), (1, 0, 128)):
        mc, mm = mgpu_model(x, y, [1, 2], G, 256, transport=transport, ozaki=0, tile=tile)
        mm.update_cache(hp)
        mu, _ = mm.split_predict(xe, xq, want_var=False)
        t = mm.timings()
        assert t["split_build"] > 0 and t["split_gemm"] > 0 and t["split_d2h"] > 0, t
        mm.close(); mc.close()
        if ref is None:
            ref = mu
        assert np.array_equal(mu, ref), (G, transport, tile)
    mu_s, _ = _single_split(gpr, x, y, hp, [1, 2], xe, xq, 0)
    cond = cond_of(cov, hp, x)
    print(f"\nsplit mean, DMMA: distributed vs single-GPU max rel {mean_err(ref, mu_s, y):.1e}, bit-identical {np.array_equal(ref, mu_s)}")
    assert mean_err(ref, mu_s, y) <= ctol(TOL_MU, cond)


@pytest.mark.parametrize("ozaki", [0, -1])
def test_mgpu_split_matches_single_gpu_n8192(gpr, ozaki):
    """Config 2 set A (N = 8192, D = 8, SE + noise) on 4 ranks against single-GPU gpr_split_predict, DMMA and the automatic route
    (INT8 eligibility of the mean products depends on the slab width there)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mg2", os.path.join(HERE, "golden", "make_golden_config2.py"))
    mg2 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg2)
    x, y, sets = mg2.inputs()
    hp = sets["A"]
    rng = np.random.default_rng(83)
    xe, xq = grid(rng, x.shape[0], 256, 2048)
    mu_s, var_s = _single_split(gpr, x, y, hp, [1, 2], xe, xq, ozaki, var_range=(1, 3))
    mc, mm = mgpu_model(x, y, [1, 2], 4, 512, ozaki=ozaki)
    mm.update_cache(hp)
    mu, var = mm.split_predict(xe, xq, var_range=(1, 3))
    mm.close(); mc.close()
    cond = _cond_bound(o.kernel((o.SE, o.NOISE), hp, x), hp[-1] ** 2 + 1e-8)
    prior = hp[0] ** 2 + hp[-1] ** 2
    em, ev = mean_err(mu, mu_s, y), np.abs(var - var_s).max() / prior
    print(f"\nsplit N = 8192 on 4 ranks, ozaki {ozaki}: cond <= {cond:.1e}, mean {em:.1e}, var {ev:.1e}")
    assert em <= ctol(TOL_MU, cond) and ev <= ctol(TOL_VAR, cond)


def test_mgpu_split_var_rows_match_mgpu_predict(gpr):
    """The var_range rows are the flattened grid points of those rows: gpr_mgpu_predict(var_diag) on them agrees; every other
    entry is exactly the prior."""
    cov = (o.SE, o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 900, 3, 1, 17)
    xe, xq = grid(rng, 3, 20, 260)
    mc, mm = mgpu_model(x, y, [1, 1, 2], 3, 128, tile=256)   # predict_tile 256 < nqp = 384: tiles of one row e x 256 / 128 q columns
    mm.update_cache(hp)
    mu, var = mm.split_predict(xe, xq, var_range=(4, 8))
    pts = np.concatenate([xe[:, e:e + 1] + xq for e in range(3, 8)], axis=1)
    _, vp, _ = mm.predict(pts, want_var=True)
    mm.close(); mc.close()
    prior = float(np.sum(hp[[0, 4, 8]] ** 2))
    v2 = var.reshape(20, 260)
    assert np.abs(v2[3:8].ravel() - vp).max() <= ctol(TOL_VAR, cond_of(cov, hp, x)) * prior
    assert np.all(v2[:3] == prior) and np.all(v2[8:] == prior)


def test_mgpu_split_errors_and_repeat(gpr):
    from gpr_sm100a import _ffi
    x, y, hp, rng = problem((o.SE, o.NOISE), 500, 2, 1, 3)
    xe, xq = grid(rng, 2, 10, 40)
    mc, mm = mgpu_model(x, y, [1, 2], 2, 128)
    L = _ffi.lib()
    GPR_ERR_ARG, GPR_ERR_STATE, GPR_ERR_UNSUPPORTED = -1, -4, -5
    mean, var = np.empty((10, 40), order="F"), np.empty(400)

    def rc(h=None, xe_=xe, ne=10, xq_=xq, nq=40, lo=1, hi=3, mean_=mean, var_=var):
        return L.gpr_mgpu_split_predict(h or mm.handle, None if xe_ is None else _ffi.dptr(xe_), ne, None if xq_ is None else _ffi.dptr(xq_),
                                        nq, lo, hi, None if mean_ is None else _ffi.dptr(mean_), None if var_ is None else _ffi.dptr(var_))

    assert rc() == GPR_ERR_STATE                                  # no evaluation yet
    mm.nlml_grad(hp, want_g=False)
    assert rc() == GPR_ERR_STATE                                  # loss-only evaluation: no inverse
    mm.update_cache(hp)
    assert rc() == 0
    for bad in (dict(lo=0), dict(hi=11), dict(lo=5, hi=3), dict(xe_=None), dict(xq_=None), dict(mean_=None), dict(ne=0), dict(nq=0)):
        assert rc(**bad) == GPR_ERR_ARG, bad
    assert rc(lo=0, var_=None) == 0                               # var_range is not looked at without var
    assert rc(lo=4, hi=3) == 0                                    # empty var_range
    K0 = mm.fetch(_ffi.FETCH_KINV)
    a = mm.split_predict(xe, xq, var_range=(2, 10))
    b = mm.split_predict(xe, xq, var_range=(2, 10))
    assert all(np.array_equal(u, v) for u, v in zip(a, b))
    assert np.array_equal(mm.fetch(_ffi.FETCH_KINV), K0)
    t = mm.timings()
    assert t["pred_kstar"] > 0 and t["pred_trsm"] > 0 and t["pred_rownorm"] > 0 and t["pred_mean"] > 0, t
    with pytest.raises(gpr.PosDefException):
        mm.update_cache(hp, eps=-10.0)                            # K - 10 I is not positive definite
    assert rc() == GPR_ERR_STATE                                  # failed factorization
    mm.close(); mc.close()
    # matrix y: no split prediction (Diagonal(wt) needs a vector, src/split_predict.jl:13)
    x3, y3, hp3, _ = problem((o.SE, o.NOISE), 300, 2, 3, 4)
    mc3, mm3 = mgpu_model(x3, y3, [1, 2], 2, 128)
    mm3.update_cache(hp3)
    assert rc(h=mm3.handle) == GPR_ERR_UNSUPPORTED
    mm3.close(); mc3.close()


def test_mgpu_split_python_mirror_end_to_end(gpr):
    """predict_mean_ / predict_ with a Cmap on MultiGPUPredictCache, into caller-owned arrays (written in place) and into arrays
    that need a copy, against GPRSplitPredictCache with the same var_range."""
    cov = (o.SE, o.NOISE)
    x, y, hp, rng = problem(cov, 800, 3, 1, 29)
    md = gpr.GPRModel(to_gpr_cov(gpr, cov), hp, x, y)
    xe, xq = grid(rng, 3, 30, 200)
    cm = gpr.Cmap(np.add, xe, xq)
    ref = gpr.GPRSplitPredictCache(md, cm, var_range=(2, 5))
    gpr.update_cache_(ref, md)
    mu_r, S_r = np.empty((30, 200), order="F"), gpr.Diagonal(np.empty(6000))
    gpr.predict_(mu_r, S_r, md, cm, ref)
    ref.close()
    pc = gpr.MultiGPUPredictCache(md, devices=_devices(3), nb=128, var_range=(2, 5))
    assert gpr.MultiGPUPredictCache(md, devices=_devices(1), nb=128).var_range == (1, 3)
    gpr.update_cache_(pc, md)
    mu0 = np.empty((30, 200), order="F")
    gpr.predict_mean_(mu0, md, cm, pc)
    mu, S = np.empty((30, 200), order="F"), gpr.Diagonal(np.empty(6000))
    ptr = (mu.ctypes.data, S.diag.ctypes.data)
    gpr.predict_(mu, S, md, cm, pc)
    assert (mu.ctypes.data, S.diag.ctypes.data) == ptr
    mu_c = np.empty((30, 200))                                    # C order: filled through a copy
    S_c = gpr.Diagonal(np.empty(6000))
    gpr.predict_(mu_c, S_c, md, cm, pc)
    pc.close()
    assert np.array_equal(mu0, mu) and np.array_equal(mu_c, mu) and np.array_equal(S_c.diag, S.diag)
    cond = cond_of(cov, hp, x)
    prior = float(np.sum(hp[[0, -1]] ** 2))
    assert mean_err(mu, mu_r, y) <= ctol(TOL_MU, cond)
    assert np.abs(S.diag - S_r.diag).max() <= ctol(TOL_VAR, cond) * prior
    assert np.all(S.diag.reshape(30, 200)[[0] + list(range(5, 30))] == prior)
